"""MatShell callbacks of the mini-app on the `/gpu/b200` backend.

Mirrors /root/reference/src/matops.c function for function:
  ApplyLocalCeedOp :26-60, FormResidual_Ceed :63-79, ApplyJacobianCoarse_Ceed :82-95,
  ApplyJacobian_Ceed :98-112, Prolong_Ceed :115-157, Restrict_Ceed :160-203, GetDiag_Ceed :206-244
and the context structs UserMult (/root/reference/elasticity.h:173-189, src/misc.c:26-70) and
UserMultProlongRestr (elasticity.h:202-215, src/misc.c:73-146).

PETSc is not available here; `LevelDM` stands in for the DM of one multigrid level: it owns
the local (L-vector: owned + ghost + Dirichlet dofs, interlaced [node][3]) and global (owned,
unconstrained dofs) layouts and performs DMGlobalToLocal / DMLocalToGlobal.  PETSc Vecs are
torch float64 tensors (device tensors for `-memtype device`, host tensors for `-memtype host`).
All device arithmetic is done by libceed_b200.so kernels.
"""
from dataclasses import dataclass

import numpy as np
import torch

from . import ceed as libceed
from .ceed import MEM_DEVICE, MEM_HOST, USE_POINTER, b2, lib


# halo/compute overlap pays once the interior kernel is long enough to hide the exchange behind (two extra
# launches, two stream hand-overs): below this many interior elements the plain sequence is used
OVERLAP_MIN_INTERIOR = 60000


class LevelDM:
    """DM stand-in for one level (degree p) of a (brick of a) box mesh.

    bc_faces: "all" (the `-test` marker label, setupdm.c:160-170), an iterable of (axis, side)
    or None.  `halo`: a ceedpetscsolid_b200.halo.Halo for partitioned runs, else None.
    """

    def __init__(self, mesh, degree, bc_faces="all", halo=None, device="cuda", node_perm=None, shared=False,
                 masked=False):
        """masked=True: "global" vectors have the LOCAL layout (every local dof, interface copies included) and the
        Dirichlet dofs are carried along as entries that are always exactly zero -- rows and columns of constrained
        dofs are masked instead of compressed out.  DMGlobalToLocal / DMLocalToGlobal then move no data at all: the
        operator reads X and accumulates into Y directly (one small kernel zeroes the Dirichlet rows of Y), which
        removes two full passes over the vectors from every MatMult.  Krylov iterates are unchanged: zero entries
        do not contribute to inner products and stay zero under the masked operator, Jacobi and the transfers.
        shared=True (partitioned runs): "global" vectors keep a consistent copy of every interface dof on
        every rank that holds it, so DMGlobalToLocal needs no communication and DMLocalToGlobal(ADD) is ONE
        symmetric sum-and-share exchange instead of two one-directional ones; `dot_weight` (1/#ranks holding
        the dof) makes inner products count each dof once."""
        self.mesh, self.degree, self.halo = mesh, degree, halo
        self.masked = bool(masked)
        self.shared = bool((shared or masked) and halo is not None)
        self.device = torch.device(device)
        nn = mesh.num_nodes(degree)
        self.lsize = 3 * nn
        bc_nodes = mesh.boundary_mask(degree, bc_faces) if bc_faces is not None else np.zeros(nn, bool)
        owned_nodes = halo.owned_node_mask if (halo is not None and not self.shared) else np.ones(nn, bool)
        free_owned = (~bc_nodes) & owned_nodes
        if node_perm is not None:  # local numbering is a permutation of the lexicographic one
            fo = np.zeros(nn, bool); fo[node_perm] = free_owned
            bc = np.zeros(nn, bool); bc[node_perm] = bc_nodes
            free_owned, bc_nodes = fo, bc
        self.bc_nodes = bc_nodes
        free_idx = np.flatnonzero(np.repeat(free_owned, 3)).astype(np.int32)
        bc_idx = np.flatnonzero(np.repeat(bc_nodes, 3)).astype(np.int32)
        fo_idx = np.arange(self.lsize, dtype=np.int32) if self.masked else free_idx
        self.nglobal = fo_idx.size
        self.free_owned_idx = torch.from_numpy(fo_idx).to(self.device)
        l2g = np.full(self.lsize, -1, dtype=np.int32)  # local dof -> global dof (-1: ghost or Dirichlet)
        l2g[free_idx] = free_idx if self.masked else np.arange(free_idx.size, dtype=np.int32)
        self.local_to_global_idx = torch.from_numpy(l2g).to(self.device)
        self.dot_weight = None
        self.n_unconstrained_local = float(free_idx.size)  # this rank's share of the global unconstrained dofs
        if self.shared:
            w = np.repeat(1.0 / halo.rank_multiplicity, 3)
            self.n_unconstrained_local = float(w[free_idx].sum())
            self.dot_weight = torch.from_numpy(w[fo_idx]).to(self.device)
        self.bc_idx = torch.from_numpy(bc_idx).to(self.device)
        self._fo_host, self._bc_host, self._free_host = fo_idx, bc_idx, free_idx

    # ---- Vec creation (DMCreateGlobalVector / DMCreateLocalVector)
    def create_global_vector(self, mem=MEM_DEVICE):
        return torch.zeros(self.nglobal, dtype=torch.float64,
                           device=self.device if mem == MEM_DEVICE else "cpu",
                           pin_memory=(mem == MEM_HOST and torch.cuda.is_available()))

    def create_local_vector(self, mem=MEM_DEVICE):
        return torch.zeros(self.lsize, dtype=torch.float64,
                           device=self.device if mem == MEM_DEVICE else "cpu",
                           pin_memory=(mem == MEM_HOST and torch.cuda.is_available()))

    # ---- DMGlobalToLocal(INSERT_VALUES) / DMLocalToGlobal(ADD_VALUES) (matops.c:33,57)
    def zero_constrained(self, X):
        """masked layouts: zero the Dirichlet entries of a "global" vector (no-op otherwise: they are not stored)"""
        if not self.masked or self.bc_idx.numel() == 0:
            return
        if X.is_cuda:
            b2(lib.b200_mask_zero(X.data_ptr(), self.bc_idx.data_ptr(), self.bc_idx.numel()))
        else:
            X.numpy()[self._bc_host] = 0.0

    def fix_diagonal(self, D):
        """masked layouts: unit diagonal on the Dirichlet rows (the masked operator has zero rows there)"""
        if not self.masked or self.bc_idx.numel() == 0:
            return
        D[self.bc_idx.long()] = 1.0

    def global_to_local(self, X, Xloc):
        if self.masked:       # free dofs only: the Dirichlet entries of Xloc (boundary values) are left alone
            if Xloc.is_cuda:
                b2(lib.b200_copy_where(Xloc.data_ptr(), X.data_ptr(), self.local_to_global_idx.data_ptr(), self.lsize))
            else:
                Xloc.numpy()[self._free_host] = X.numpy()[self._free_host]
            return
        if Xloc.is_cuda:
            b2(lib.b200_scatter_set(Xloc.data_ptr(), self.free_owned_idx.data_ptr(), X.data_ptr(), self.nglobal))
        else:
            Xloc.numpy()[self._fo_host] = X.numpy()
        if self.halo is not None and not self.shared:
            self.halo.owner_to_ghost(Xloc)

    def zero_and_global_to_local(self, X, Xloc):
        """VecZeroEntries(Xloc) followed by DMGlobalToLocal(INSERT_VALUES) (matops.c:106 + :33) in one
        pass over Xloc (device vectors); identical result, one third of the memory traffic."""
        if Xloc.is_cuda:
            b2(lib.b200_gather_or_zero(Xloc.data_ptr(), X.data_ptr(), self.local_to_global_idx.data_ptr(), self.lsize))
            if self.halo is not None and not self.shared:
                self.halo.owner_to_ghost(Xloc)
        else:
            Xloc.zero_()
            self.global_to_local(X, Xloc)

    def local_to_global(self, Yloc, Y, exchange=True):
        """VecZeroEntries(Y); DMLocalToGlobal(dm, Yloc, ADD_VALUES, Y): constrained dofs dropped.
        exchange=False: the interface entries of Yloc are already complete on every rank (injected prolongation)."""
        if self.halo is not None and (exchange or not self.shared):
            if self.shared:
                self.halo.sum_and_share(Yloc)
            else:
                self.halo.ghost_to_owner_add(Yloc)
        if self.masked:
            if Y.data_ptr() != Yloc.data_ptr():
                Y.copy_(Yloc)
            self.zero_constrained(Y)
            return
        if Yloc.is_cuda:
            b2(lib.b200_gather(Y.data_ptr(), Yloc.data_ptr(), self.free_owned_idx.data_ptr(), self.nglobal))
        else:
            Y.numpy()[:] = Yloc.numpy()[self._fo_host]

    def make_consistent(self, X):
        """shared layouts: replace every copy of an interface dof by the average of the copies"""
        if not self.shared:
            self.zero_constrained(X)
            return
        Xl = self.create_local_vector(MEM_DEVICE if X.is_cuda else MEM_HOST)
        X.mul_(self.dot_weight)
        self.global_to_local(X, Xl)
        self.local_to_global(Xl, X)

    def insert_boundary_values(self, Xloc, values):
        """DMPlexInsertBoundaryValues stand-in: values = tensor over bc dofs (or None = zero)."""
        if values is None:
            return
        if Xloc.is_cuda:
            b2(lib.b200_scatter_set(Xloc.data_ptr(), self.bc_idx.data_ptr(), values.data_ptr(), self.bc_idx.numel()))
        else:
            Xloc.numpy()[self._bc_host] = values.cpu().numpy()


@dataclass
class UserMult:
    """elasticity.h:173-189; wired by SetupJacobianCtx (src/misc.c:26-70)."""
    dm: LevelDM
    Xloc: torch.Tensor
    Yloc: torch.Tensor
    Xceed: object
    Yceed: object
    op: object
    qf: object
    ceed: object
    phys: object = None
    physSmoother: object = None
    memType: int = MEM_DEVICE
    loadIncrement: float = 1.0
    bc_values: object = None  # callable(loadIncrement) -> tensor over dm.bc_idx, or None
    overlap: bool = True      # partitioned + masked layout: overlap the halo exchange with the interior elements
    fused: object = None      # cached CeedOperatorIsFusedB200(op)


def setup_jacobian_ctx(dm, ceed, data, phys, physSmoother=None, memType=MEM_DEVICE):
    """SetupJacobianCtx (src/misc.c:26-70)."""
    return UserMult(dm=dm, Xloc=dm.create_local_vector(memType), Yloc=dm.create_local_vector(memType),
                    Xceed=data.xceed, Yceed=data.yceed, op=data.opJacob, qf=data.qfJacob, ceed=ceed, phys=phys,
                    physSmoother=physSmoother, memType=memType)


def ApplyLocalCeedOp(X, Y, user, zero_xloc=False):
    """matops.c:26-60: Y = P^T A_loc P X.  zero_xloc fuses the caller's VecZeroEntries(Xloc)
    (ApplyJacobian_Ceed, matops.c:106) into the global-to-local pass."""
    dm = user.dm
    if dm.masked and zero_xloc:
        # masked layout: X already IS the L-vector with zero boundary values and Y the L-vector to accumulate
        # into -- no DMGlobalToLocal / DMLocalToGlobal data movement at all
        user.Xceed.set_array(X, user.memType, USE_POINTER)
        user.Yceed.set_array(Y, user.memType, USE_POINTER)
        if user.fused is None:
            # built-in fused kernels and K12 (the fused kernel around a JIT-compiled user QFunction) both take the
            # one-call partitioned apply
            user.fused = bool(user.op.is_fused or user.op.is_jit_fused)
        if X.is_cuda and user.fused and (dm.halo is None or dm.halo.handle is not None):
            # the whole MatMult in one C call: zero Y, interface elements, peer-memory halo exchange overlapped with
            # the interior elements, ordered sum of the holders' partial sums, zero the Dirichlet rows
            nif = dm.mesh.n_interface if (dm.halo is not None and user.overlap) else 0
            user.op.apply_partitioned(user.Xceed, user.Yceed, nif, dm.halo.handle if dm.halo is not None else None,
                                      dm.bc_idx)
            user.Xceed.take_array(user.memType)
            user.Yceed.take_array(user.memType)
            return
        nif = dm.mesh.n_interface if dm.halo is not None else 0
        if (nif and user.overlap and X.is_cuda and dm.mesh.nelem - nif >= OVERLAP_MIN_INTERIOR
                and not user.ceed.is_deterministic):   # the ordered sum runs over the whole restriction
            # partitioned: the elements touching a partition interface come first in the element numbering;
            # once they are done every shared dof holds its complete partial sum, so the halo exchange runs
            # (side stream, NCCL) while the interior elements are processed
            user.Yceed.set_value(0.0)
            user.op.apply_add_range(user.Xceed, user.Yceed, 0, nif)
            dm.halo.sum_and_share_begin(Y)
            user.op.apply_add_range(user.Xceed, user.Yceed, nif, dm.mesh.nelem)
            dm.halo.sum_and_share_end(Y)
            user.Xceed.take_array(user.memType)
            user.Yceed.take_array(user.memType)
            dm.zero_constrained(Y)
            return
        user.op.apply(user.Xceed, user.Yceed)
        user.Xceed.take_array(user.memType)
        user.Yceed.take_array(user.memType)
        dm.local_to_global(Y, Y)        # halo sum-and-share (partitioned runs) + zero the Dirichlet rows, in place
        return
    if zero_xloc:
        user.dm.zero_and_global_to_local(X, user.Xloc)            # :106 + :33
    else:
        user.dm.global_to_local(X, user.Xloc)                     # :33
    # :34 VecZeroEntries(Yloc) is subsumed: CeedOperatorApply zeroes its output vector itself
    user.Xceed.set_array(user.Xloc, user.memType, USE_POINTER)    # :40
    user.Yceed.set_array(user.Yloc, user.memType, USE_POINTER)    # :41
    user.op.apply(user.Xceed, user.Yceed)                         # :46
    user.Xceed.take_array(user.memType)                           # :49
    user.Yceed.take_array(user.memType)                           # :50
    user.dm.local_to_global(user.Yloc, Y)                         # :56-57


def FormResidual_Ceed(X, Y, user):
    """matops.c:63-79: boundary values at `loadIncrement`, then the residual operator
    (which also rewrites gradu for the following Jacobian applies)."""
    user.Xloc.zero_()
    if user.bc_values is not None:
        user.dm.insert_boundary_values(user.Xloc, user.bc_values(user.loadIncrement))
    ApplyLocalCeedOp(X, Y, user)


def ApplyJacobian_Ceed(user, X, Y):
    """matops.c:98-112 (and ApplyJacobianCoarse_Ceed :82-95): zero boundary values, apply."""
    ApplyLocalCeedOp(X, Y, user, zero_xloc=True)


def GetDiag_Ceed(user, D):
    """matops.c:206-244."""
    if user.physSmoother is not None:
        user.qf.set_context(user.physSmoother)
    user.Xceed.set_array(user.Xloc, user.memType, USE_POINTER)
    user.op.linear_assemble_diagonal(user.Xceed)
    if user.physSmoother is not None:
        user.qf.set_context(user.phys)
    user.Xceed.take_array(user.memType)
    user.dm.local_to_global(user.Xloc, D)
    user.dm.fix_diagonal(D)
    user.Xloc.zero_()


def _state_lvector(X, user):
    """Xloc = [free dofs of X; boundary values at user.loadIncrement] (VecZeroEntries, DMGlobalToLocal,
    DMPlexInsertBoundaryValues: matops.c:258-262, misc.c:243-247)."""
    user.dm.zero_and_global_to_local(X, user.Xloc)
    if user.bc_values is not None:
        user.dm.insert_boundary_values(user.Xloc, user.bc_values(user.loadIncrement))
    return user.Xloc


def ComputeStrainEnergy(user, opEnergy, X, dist=None):
    """matops.c:247-300: strain energy of the state X = sum of the entries of E_e^T B_e^T [w detJ psi] (one scalar
    per mesh node), summed over ranks."""
    xloc = _state_lvector(X, user)
    nn = user.dm.lsize // 3
    eloc = user.ceed.Vector(nn)
    user.Xceed.set_array(xloc, user.memType, USE_POINTER)
    opEnergy.apply(user.Xceed, eloc)
    user.Xceed.take_array(user.memType)
    energy = float(eloc.to_numpy().sum())          # CeedVectorGetArrayRead(HOST) + host loop, matops.c:285-290
    eloc.destroy()
    if dist is not None and dist.get_world_size() > 1:
        t = torch.tensor([energy], dtype=torch.float64, device=user.dm.device)
        dist.all_reduce(t)
        energy = float(t.item())
    return energy


def ComputeDiagnosticQuantities(user, opDiagnostic, ErestrictDiagnostic, X, halo8=None):
    """ViewDiagnosticQuantities (src/misc.c:217-300) without the VTK writer: nodal (u, pressure, two strain
    invariants, volume ratio, energy density), element contributions summed and divided by the node multiplicity.
    halo8: a Halo built with ncomp=8 for partitioned runs (interface nodes get contributions from every rank).
    Returns a (nodes, 8) tensor on the level's device."""
    xloc = _state_lvector(X, user)
    nn = user.dm.lsize // 3
    yloc = torch.zeros(8 * nn, dtype=torch.float64, device=xloc.device)
    mult = torch.zeros_like(yloc)
    yc = user.ceed.Vector(8 * nn)
    user.Xceed.set_array(xloc, user.memType, USE_POINTER)
    yc.set_array(yloc, user.memType, USE_POINTER)
    opDiagnostic.apply(user.Xceed, yc)
    user.Xceed.take_array(user.memType)
    yc.take_array(user.memType)
    yc.set_array(mult, user.memType, USE_POINTER)
    ErestrictDiagnostic.get_multiplicity(yc)
    yc.take_array(user.memType)
    yc.destroy()
    if halo8 is not None:
        halo8.sum_and_share(yloc)
        halo8.sum_and_share(mult)
    return (yloc / mult).reshape(nn, 8)


@dataclass
class UserMultProlongRestr:
    """elasticity.h:202-215; SetupProlongRestrictCtx (src/misc.c:73-146)."""
    dmC: LevelDM
    dmF: LevelDM
    locVecC: torch.Tensor
    locVecF: torch.Tensor
    multVec: torch.Tensor
    ceedVecC: object
    ceedVecF: object
    opProlong: object
    opRestrict: object
    ceed: object
    memType: int = MEM_DEVICE
    fusedScale: object = None   # CeedVector of multVec handed to the fused transfer kernels (None: separate passes)
    inject: bool = False        # prolongation stores the interpolant (complete, to rounding, on every holder of a node)


def setup_prolong_restrict_ctx(dmC, dmF, ceed, dataC, dataF, userC, userF, memType=MEM_DEVICE, fuse_scaling=True):
    """src/misc.c:73-146: shares the level work vectors; multVec = 1 / multiplicity of the fine
    restriction, summed over ranks (L2G then G2L) before the reciprocal (:115-143)."""
    mult_ceed = dataF.Erestrictu.create_vector()
    dataF.Erestrictu.get_multiplicity(mult_ceed)
    mult = torch.from_numpy(mult_ceed.to_numpy())
    mult_ceed.destroy()
    mult = mult.to(dmF.device) if memType == MEM_DEVICE else mult
    if dmF.halo is not None:
        if dmF.shared:
            dmF.halo.sum_and_share(mult)
        else:
            dmF.halo.ghost_to_owner_add(mult)
            dmF.halo.owner_to_ghost(mult)
    multVec = torch.where(mult > 0, 1.0 / mult, mult)
    fused = None
    if fuse_scaling and memType == MEM_DEVICE and dataF.opProlong.is_fused and dataF.opRestrict.is_fused:
        # the fused transfer kernels apply multVec themselves: no VecPointwiseMult passes (matops.c:149,176), and
        # the prolongation stores the interpolant at every fine node (no atomics, no pre-zeroed output)
        fused = ceed.Vector(multVec.numel())
        fused.set_array(multVec, MEM_DEVICE, USE_POINTER)
        # owner/ghost layouts ADD the ghost copies into the owner afterwards: they need partial sums, not complete values.
        # The injected value is the same at every holder of a node only to the last bit: elements sharing it with other
        # local axes contract in another order, and the last store wins.  Deterministic mode therefore sums the scaled
        # element copies in a fixed order (and, partitioned, exchanges them like every other operator).
        inject = (dmF.halo is None or dmF.shared) and not ceed.is_deterministic
        dataF.opProlong.set_transfer_scaling(fused, inject=inject)
        dataF.opRestrict.set_transfer_scaling(fused)
    return UserMultProlongRestr(dmC=dmC, dmF=dmF, locVecC=userC.Xloc, locVecF=userF.Xloc, multVec=multVec,
                                ceedVecC=dataC.xceed, ceedVecF=dataF.xceed, opProlong=dataF.opProlong,
                                opRestrict=dataF.opRestrict, ceed=ceed, memType=memType, fusedScale=fused,
                                inject=fused is not None and inject)


def _pointwise_mult(w, x, y):
    if w.is_cuda:
        b2(lib.b200_vec_pointwise_mult(w.data_ptr(), x.data_ptr(), y.data_ptr(), w.numel()))
    else:
        torch.mul(x, y, out=w)


def Prolong_Ceed(user, X, Y):
    """matops.c:115-157."""
    user.locVecC.zero_()
    user.dmC.global_to_local(X, user.locVecC)
    if user.fusedScale is not None:
        # scaling inside the kernel; injected: every fine node is overwritten with the interpolant, complete on every
        # rank that holds it -> no zeroing, no pointwise product, no halo sum
        user.ceedVecC.set_array(user.locVecC, user.memType, USE_POINTER)
        user.ceedVecF.set_array(user.locVecF, user.memType, USE_POINTER)
        if user.inject:
            user.opProlong.apply_add(user.ceedVecC, user.ceedVecF)
        else:
            user.opProlong.apply(user.ceedVecC, user.ceedVecF)
        user.ceedVecC.take_array(user.memType)
        user.ceedVecF.take_array(user.memType)
        user.dmF.local_to_global(user.locVecF, Y, exchange=not user.inject)
        return
    user.locVecF.zero_()
    user.ceedVecC.set_array(user.locVecC, user.memType, USE_POINTER)
    user.ceedVecF.set_array(user.locVecF, user.memType, USE_POINTER)
    user.opProlong.apply(user.ceedVecC, user.ceedVecF)
    user.ceedVecC.take_array(user.memType)
    user.ceedVecF.take_array(user.memType)
    _pointwise_mult(user.locVecF, user.locVecF, user.multVec)     # :149
    user.dmF.local_to_global(user.locVecF, Y)


def Restrict_Ceed(user, X, Y):
    """matops.c:160-203."""
    user.locVecF.zero_()
    user.dmF.global_to_local(X, user.locVecF)
    user.locVecC.zero_()
    if user.fusedScale is None:
        _pointwise_mult(user.locVecF, user.locVecF, user.multVec)     # :176 (else: inside the fused kernel)
    user.ceedVecF.set_array(user.locVecF, user.memType, USE_POINTER)
    user.ceedVecC.set_array(user.locVecC, user.memType, USE_POINTER)
    user.opRestrict.apply(user.ceedVecF, user.ceedVecC)
    user.ceedVecF.take_array(user.memType)
    user.ceedVecC.take_array(user.memType)
    user.dmC.local_to_global(user.locVecC, Y)
