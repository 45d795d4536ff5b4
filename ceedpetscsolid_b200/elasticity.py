"""The mini-app driver on the `/gpu/b200` backend: what /root/reference/elasticity.c `main` does
between CeedInit (:110) and the end of the load-increment loop (:676), for synthetic box meshes and unstructured
hex8 meshes, on one GPU or partitioned over several.

  set-up           elasticity.c:132-281  -> setuplibceed.setup_all, matops.LevelDM per level
  MatShell ctxs    elasticity.c:386-452  -> matops.setup_jacobian_ctx / setup_prolong_restrict_ctx
  solver config    elasticity.c:498-603  -> solver.PMultigrid + solver.pcg
  solve            elasticity.c:632-676  -> solver.newton_solve
  clamp BCs        src/boundary.c:53-74  -> bc_clamp (same expression, including its precedence quirk)
"""
import math
from dataclasses import dataclass, field

import numpy as np
import torch

from . import ceed as libceed
from . import matops, setuplibceed, solver
from .mesh import BoxMesh, grid_for


def bc_mms(coords, load):
    """BCMMS (src/boundary.c:31-45): the manufactured solution on the boundary."""
    x, y, z = coords[:, 0], coords[:, 1], coords[:, 2]
    u = np.empty_like(coords)
    u[:, 0] = np.exp(2 * x) * np.sin(3 * y) * np.cos(4 * z) / 1e8 * load
    u[:, 1] = np.exp(3 * y) * np.sin(4 * z) * np.cos(2 * x) / 1e8 * load
    u[:, 2] = np.exp(4 * z) * np.sin(2 * x) * np.cos(3 * y) / 1e8 * load
    return u


def bc_clamp(coords, load, clamp):
    """BCClamp (src/boundary.c:53-74): clamp = [tx,ty,tz, kx,ky,kz, theta/pi] (translate, axis, rotation)."""
    x, y, z = coords[:, 0], coords[:, 1], coords[:, 2]
    lx, ly, lz = (clamp[i] * load for i in range(3))
    kx, ky, kz = clamp[3], clamp[4], clamp[5]
    theta = clamp[6] * math.pi * load
    c, s = math.cos(theta), math.sin(theta)
    u = np.empty_like(coords)
    u[:, 0] = lx + s * (-kz * y + ky * z) + (1 - c) * (-ky * ky + kz * kz * x + kx * ky * y + kx * kz * z)
    u[:, 1] = ly + s * (kz * x + -kx * z) + (1 - c) * (kx * ky * x - (kx * kx + kz * kz) * y + ky * kz * z)
    u[:, 2] = lz + s * (-ky * x + kx * y) + (1 - c) * (kx * kz * x + ky * kz * y - (kx * kx + ky * ky) * z)
    return u


@dataclass
class AppCtx:
    """The options of /root/reference/src/cloptions.c that matter here."""
    problem: str = "hyperFS"
    degree: int = 4
    n: tuple = (8, 8, 8)
    nu: float = 0.3
    E: float = 1.0
    qextra: int = 0
    multigrid: str = "logarithmic"
    num_steps: int = 10
    perturb: float = 0.0
    forcing: str = "none"          # -forcing none|constant|mms
    forcing_vector: tuple = (0.0, -1.0, 0.0)
    test_mode: bool = False        # -test: MMS forcing, BCMMS on every boundary face (cloptions.c:185-187, setupdm.c:160-170)
    # clamped faces: (axis, side) -> [tx,ty,tz, kx,ky,kz, theta/pi]  (-bc_clamp, -bc_clamp_N_translate/_rotate)
    clamp: dict = field(default_factory=lambda: {(2, 0): [0, 0, 0, 0, 0, 1, 0], (2, 1): [0, 0, -0.1, 0, 0, 1, 0]})
    # -mesh file.exo (setupdm.c:40-68): an exodus.HexMesh; `clamp` is then keyed by side-set id (-bc_clamp 998,999)
    mesh: object = None


def build_h_dms(gmesh, grid, rank, world, faces, device, dist=None, min_elems=2, masked=False):
    """LevelDMs (degree 1) of successively halved box meshes below the p = 1 level, for the h-multigrid coarse
    solve.  Halving stops when a brick would have an odd element count or fewer than `min_elems` per axis."""
    dms = []
    n = gmesh.n
    while all(v % (2 * grid[d]) == 0 and v // (2 * grid[d]) >= min_elems for d, v in enumerate(n)):
        n = tuple(v // 2 for v in n)
        gm = BoxMesh(n=n, lengths=gmesh.lengths)
        mesh = gm.brick(grid, rank) if world > 1 else gm
        halo = None
        if world > 1:
            from .halo import Halo
            halo = Halo(gm, grid, rank, 1, dist, device=device if isinstance(device, str) and device == "cpu" else None)
        dms.append(matops.LevelDM(mesh, 1, bc_faces=faces, halo=halo, device=device, shared=True, masked=masked))
    return dms


class GpuLevel:
    """One p-multigrid level on the /gpu/b200 backend (the MatShell of elasticity.c:392-411)."""

    def __init__(self, dm, user, res_user=None):
        self.dm, self.user, self.res_user = dm, user, res_user
        self.n, self.device = dm.nglobal, dm.device

    def jacobian(self, X, Y):
        matops.ApplyJacobian_Ceed(self.user, X, Y)

    def diagonal(self, D):
        matops.GetDiag_Ceed(self.user, D)

    coo = None

    def enable_coo(self, ceed, mesh):
        """Coarse (trilinear) level: assemble element matrices with CeedOperatorLinearAssemble (one pass over the
        Jacobian cache) instead of colouring the operator (misc.c:151-183)."""
        level = self

        class _Coo:
            elem_nodes = torch.from_numpy(mesh.offsets(1).reshape(-1, 8) // 3).to(self.device)
            vals = torch.zeros(elem_nodes.shape[0] * 576, dtype=torch.float64, device=self.device)
            vec = ceed.Vector(vals.numel())
            deterministic = ceed.is_deterministic

            def values(self):
                self.vec.set_array(self.vals, level.user.memType)
                level.user.op.linear_assemble(self.vec)
                self.vec.take_array(level.user.memType)
                return self.vals
        self.coo = _Coo()

    def local_apply(self, xloc, yloc):
        u = self.user
        u.Xceed.set_array(xloc, u.memType)
        u.Yceed.set_array(yloc, u.memType)
        u.op.apply(u.Xceed, u.Yceed)
        u.Xceed.take_array(u.memType)
        u.Yceed.take_array(u.memType)

    def residual(self, U, F, load):
        """FormResidual_Ceed minus the (load-scaled) forcing vector: SNESSolve(snes, F_ext, U) (elasticity.c:645-654)."""
        self.res_user.loadIncrement = load
        matops.FormResidual_Ceed(U, F, self.res_user)
        if self.forcing is not None:
            solver.Vec.axpy(F, -load, self.forcing)

    forcing = None

    def bc_increment_rhs(self, F, load_prev, load):
        """F = P^T A_loc(U) [0; u_bc(load) - u_bc(load_prev)]: the Jacobian applied to the boundary increment."""
        u, r = self.user, self.res_user
        u.Xloc.zero_()
        u.dm.insert_boundary_values(u.Xloc, r.bc_values(load) - r.bc_values(load_prev))
        self.local_apply(u.Xloc, u.Yloc)
        u.dm.local_to_global(u.Yloc, F)
        if self.forcing is not None:
            solver.Vec.axpy(F, -(load - load_prev), self.forcing)


class GpuTransfer:
    def __init__(self, pr):
        self.pr = pr

    def prolong(self, Xc, Yf):
        matops.Prolong_Ceed(self.pr, Xc, Yf)

    def restrict(self, Xf, Yc):
        matops.Restrict_Ceed(self.pr, Xf, Yc)


class Elasticity:
    """Builds the whole solver stack for one rank (one GPU)."""

    def __init__(self, app, dist=None, rank=0, world=1, device_id=0, gmesh=None, coarse_rtol=1e-2, coarse="hmg",
                 assemble="coo", masked=True, overlap=True, halo="p2p", deterministic=False, amg_max_coarse=None,
                 qf_locators=None):
        """coarse: the solve on the assembled p = 1 level -- "hmg" (geometric h-multigrid on box meshes, Jacobi-PCG on
        unstructured ones), "pcg" (Jacobi-PCG) or "amg" (one V-cycle of smoothed-aggregation AMG, any mesh; with
        world > 1 every rank holds the whole hierarchy, amg.RedundantAMG, masked layout only; amg_max_coarse: rows of
        its directly solved coarsest level, default amg.MAX_COARSE_DOFS).  Unstructured meshes (app.mesh) are split
        into world parts by coordinate bisection (exodus.HexMesh.brick), box meshes into bricks.  masked: constrained
        dofs are masked in L-vector-shaped global vectors (no G2L/L2G copies, see LevelDM);
        False: compressed PETSc-style global vectors.  deterministic: "/gpu/b200:deterministic" -- every transposed
        restriction sums in the serial /cpu/self order (no FP64 atomics anywhere on the path).  qf_locators:
        {"apply": "<file>:<Name>", "jacob": "<file>:<Name>"} replaces the residual / Jacobian QFunctions of app.problem
        (same fields) by user QFunctions, compiled at set-up on the "/gpu/b200:jit" resource.  Their operators run on
        K12, the fused kernel generated around the user function (compiled at the first apply), and their diagonal on
        K14, the diagonal kernel generated around it (compiled at the first diagonal; the Jacobi / Chebyshev smoothers
        of every level call it).  The p = 1 level has no built-in Jacobian: on unstructured meshes, and with
        coarse="amg" on any mesh, its element matrices come from K13, CeedOperatorLinearAssemble around the user
        function (which must be linear in its active input, as every Jacobian QFunction is); box meshes with "hmg" or
        "pcg" assemble it by colouring.  Strain energy and diagnostics keep the problem's stock model."""
        if coarse == "amg" and world > 1:
            # checked before any device work: the redundant AMG gathers every rank's element matrices and right-hand
            # side through the process group, and exists only for the masked layout
            if not masked:
                raise NotImplementedError("coarse='amg' with world > 1 needs the masked layout (masked=True)")
            if dist is None:
                raise NotImplementedError("coarse='amg' with world > 1 runs the redundant AMG over torch.distributed: "
                                          "pass the process group (dist); without one the AMG runs on one GPU only")
        self.app, self.dist = app, dist
        halo_mode = halo
        grid = grid_for(world)
        if app.mesh is not None:
            gmesh = app.mesh
        self.gmesh = gmesh if gmesh is not None else BoxMesh(n=app.n, perturb=app.perturb, seed=0)
        self.mesh = self.gmesh.brick(grid, rank, interface_first=masked and overlap) if world > 1 else self.gmesh
        self.ceed = libceed.Ceed(f"/gpu/b200:device_id={device_id}" + (":deterministic" if deterministic else "")
                                 + (":jit" if qf_locators else ""))
        self.degrees, self.data, self.phys = setuplibceed.setup_all(self.ceed, self.mesh, app.problem, app.degree, app.nu,
                                                                    app.E, app.qextra, app.multigrid,
                                                                    qf_locators=qf_locators)
        if app.test_mode:
            app.forcing = "mms"
        faces = "all" if app.test_mode else list(app.clamp.keys())
        self.dms, self.users = [], []
        for l, deg in enumerate(self.degrees):
            halo = None
            if world > 1:
                from .halo import Halo
                halo = Halo(self.gmesh, grid, rank, deg, dist)
                if halo_mode == "p2p" and not halo.enable_p2p():
                    raise RuntimeError(f"peer-memory halo set-up failed: {halo._p2p_error}")
            dm = matops.LevelDM(self.mesh, deg, bc_faces=faces, halo=halo, device=f"cuda:{device_id}", shared=True,
                                masked=masked)
            self.dms.append(dm)
            self.users.append(matops.setup_jacobian_ctx(dm, self.ceed, self.data[l], self.phys))
        fine = len(self.degrees) - 1
        fu = self.users[fine]
        # resCtx = shallow copy of the fine Jacobian ctx with op = opApply (elasticity.c:420-425)
        self.res_user = matops.UserMult(dm=fu.dm, Xloc=fu.Xloc, Yloc=fu.Yloc, Xceed=fu.Xceed, Yceed=fu.Yceed,
                                        op=self.data[fine].opApply, qf=self.data[fine].qfApply, ceed=self.ceed,
                                        phys=self.phys, memType=fu.memType, bc_values=self._bc_values_fn(self.dms[fine], app))
        self.levels = [GpuLevel(self.dms[l], self.users[l], self.res_user if l == fine else None)
                       for l in range(len(self.degrees))]
        op0 = self.users[0].op
        unstructured = not getattr(self.gmesh, "structured", True)
        if assemble == "coo" and self.degrees[0] == 1 and (
                op0.is_fused or (op0.is_jit_fused and (unstructured or coarse == "amg"))):
            self.levels[0].enable_coo(self.ceed, self.mesh)
        self.transfers = [None]
        for l in range(1, len(self.degrees)):
            pr = matops.setup_prolong_restrict_ctx(self.dms[l - 1], self.dms[l], self.ceed, self.data[l - 1], self.data[l],
                                                   self.users[l - 1], self.users[l])
            self.transfers.append(GpuTransfer(pr))
        if app.forcing != "none":
            # global forcing vector (elasticity.c:236-245, 288-300): L-vector from the forcing operator, then L2G ADD
            floc = self.dms[fine].create_local_vector()
            fc = self.ceed.Vector(floc.numel())
            fc.set_array(floc)
            setuplibceed.setup_forcing(self.ceed, self.mesh, self.data[fine], app.forcing, self.phys, app.forcing_vector, fc)
            fc.take_array()
            fc.destroy()
            Fext = self.dms[fine].create_global_vector()
            self.dms[fine].local_to_global(floc, Fext)
            self.levels[fine].forcing = Fext
        self.V = solver.Vec(dist if world > 1 else None)
        self.V.consistent = {}
        h_dms = build_h_dms(self.gmesh, grid, rank, world, faces, f"cuda:{device_id}", dist, masked=masked) \
            if coarse == "hmg" and getattr(self.gmesh, "structured", True) else None
        if halo_mode == "p2p":
            for dm in (h_dms or []):
                if dm.halo is not None and not dm.halo.enable_p2p():
                    raise RuntimeError(f"peer-memory halo set-up failed: {dm.halo._p2p_error}")
        for dm in self.dms + list(h_dms or []):
            if dm.dot_weight is not None:
                self.V.set_weight(dm.nglobal, dm.dot_weight)
            if dm.dot_weight is not None or dm.masked:
                self.V.consistent[dm.nglobal] = dm.make_consistent
        self.all_dms = self.dms + list(h_dms or [])
        amg_solver = None
        if coarse == "amg":
            if self.levels[0].coo is None:
                raise ValueError("coarse='amg' needs the element matrices of the p = 1 level (assemble='coo', and a "
                                 "built-in fused or K12 operator there)")
            from .amg import MAX_COARSE_DOFS, RedundantAMG, SmoothedAggregationAMG
            mc = MAX_COARSE_DOFS if amg_max_coarse is None else amg_max_coarse
            if world > 1:
                amg_solver = RedundantAMG(self.dms[0], self.mesh, self.gmesh, faces, dist, max_coarse=mc)
            else:
                amg_solver = SmoothedAggregationAMG(self.dms[0], self.mesh, max_coarse=mc)
        self.pc = solver.PMultigrid(self.V, self.levels, self.transfers, coarse_rtol=coarse_rtol, h_dms=h_dms,
                                    amg=amg_solver)
        self.U = self.dms[fine].create_global_vector()

    @staticmethod
    def _bc_values_fn(dm, app):
        """DMPlexInsertBoundaryValues stand-in: clamp values at the Dirichlet nodes for a load fraction."""
        p = dm.degree
        coords = dm.mesh.node_coords(p)
        bc_nodes = np.flatnonzero(dm.bc_nodes)
        xyz = coords[bc_nodes]
        if app.test_mode:
            return lambda load: torch.from_numpy(bc_mms(xyz, load).reshape(-1)).to(dm.device)
        face_of = np.full(bc_nodes.size, -1)
        for fi, face in enumerate(app.clamp.keys()):  # later faces win on shared edges, as DMAddBoundary order
            on = dm.mesh.boundary_mask(p, [face])[bc_nodes]
            face_of[on] = fi
        clamps = list(app.clamp.values())

        def values(load):
            u = np.zeros((bc_nodes.size, 3))
            for fi, cl in enumerate(clamps):
                m = face_of == fi
                if m.any():
                    u[m] = bc_clamp(xyz[m], load, cl)
            return torch.from_numpy(u.reshape(-1)).to(dm.device)

        return values

    def solve(self, log=None, **kw):
        self.U.zero_()
        fine = self.levels[-1]
        out = solver.newton_solve(self.V, fine, self.pc, self.U, num_increments=self.app.num_steps, log=log,
                                  check=self.check_halos, **kw)
        self.check_halos()
        out["dofs_global_unconstrained"] = self._global_unconstrained()
        # "DoFs/Sec in SNES" = global dofs x total KSP iterations / solve time (elasticity.c:762-764), in MDoF/s
        out["mdofs_per_sec_in_snes"] = 1e-6 * out["dofs_global_unconstrained"] * out["ksp_its"] / max(out["time_s"], 1e-12)
        return out

    def check_halos(self):
        """Raises if a peer-memory halo exchange of any level timed out (Halo.check_p2p; synchronises)."""
        for dm in self.all_dms:
            if dm.halo is not None:
                dm.halo.check_p2p()

    def close(self):
        """Collective: release the peer-memory windows of every level."""
        for dm in self.all_dms:
            if dm.halo is not None:
                dm.halo.close()

    def strain_energy(self):
        """elasticity.c:820-830: strain energy of the current state at full load (ComputeStrainEnergy)."""
        fine = len(self.degrees) - 1
        if self.data[fine].opEnergy is None:
            setuplibceed.setup_energy(self.ceed, self.mesh, self.app.problem, self.data[fine], self.phys)
        self.res_user.loadIncrement = 1.0
        return matops.ComputeStrainEnergy(self.res_user, self.data[fine].opEnergy, self.U,
                                          self.dist if self.dist is not None and self.dist.get_world_size() > 1 else None)

    def diagnostic_quantities(self):
        """elasticity.c:836-850 (ViewDiagnosticQuantities without the VTK writer): (local nodes, 8) tensor =
        displacement, pressure, two strain invariants, volume ratio, energy density."""
        fine = len(self.degrees) - 1
        d = self.data[fine]
        if d.opDiagnostic is None:
            setuplibceed.setup_diagnostic(self.ceed, self.mesh, self.app.problem, d, self.phys)
        halo8 = None
        if self.dms[fine].halo is not None:
            from .halo import Halo
            h = self.dms[fine].halo
            halo8 = Halo(self.gmesh, h.grid, h.rank, h.p, h.dist, ncomp=8)
        self.res_user.loadIncrement = 1.0
        return matops.ComputeDiagnosticQuantities(self.res_user, d.opDiagnostic, d.ErestrictDiagnostic, self.U, halo8)

    def mms_l2_error(self):
        """elasticity.c:770-816: |U - U_true| / |U| over the global (unconstrained) dofs."""
        fine = len(self.degrees) - 1
        true_l = setuplibceed.setup_true_solution(self.ceed, self.mesh, self.data[fine], self.degrees[fine] + 1)
        dm = self.dms[fine]
        tg = torch.from_numpy(true_l).to(dm.device)[dm.free_owned_idx.long()]
        dm.zero_constrained(tg)
        err2, u2 = self.V.dot(self.U - tg, self.U - tg), self.V.dot(self.U, self.U)
        return math.sqrt(err2 / u2)

    def _global_unconstrained(self):
        dm = self.dms[-1]
        n = torch.tensor([dm.n_unconstrained_local], dtype=torch.float64, device=dm.device)
        if self.dist is not None and self.dist.get_world_size() > 1:
            self.dist.all_reduce(n)
        return int(round(n.item()))
