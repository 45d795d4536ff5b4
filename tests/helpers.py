"""Shared test set-up: synthetic box problems (SURVEY.md 8(d)) evaluated with the oracle."""
import numpy as np

from ceedpetscsolid_b200.mesh import BoxMesh, smooth_displacement
from oracle import oracle

PHYS = (0.3, 1.0)  # nu, E  (TESTARGS, /root/reference/elasticity.c:36)


class OracleProblem:
    """Box problem at fine degree `p` with level degree `pl` (P = pl+1, Q = p+1+qextra)."""

    def __init__(self, problem, n, p, pl=None, perturb=0.08, qextra=0, scale=0.02, which=None,
                 node_perm_seed=None, mesh=None):
        self.problem, self.p, self.pl = problem, p, (p if pl is None else pl)
        self.which = which
        n = (n, n, n) if np.isscalar(n) else n
        self.mesh = mesh if mesh is not None else BoxMesh(n=n, perturb=perturb, seed=0)
        self.nelem = self.mesh.nelem
        self.P, self.Pf, self.Q = self.pl + 1, p + 1, p + 1 + qextra
        self.perm = None
        if node_perm_seed is not None:
            self.perm = np.random.default_rng(node_perm_seed).permutation(self.mesh.num_nodes(self.pl))
        self.offsets = self.mesh.offsets(self.pl, node_perm=self.perm)
        self.offsets_fine = self.mesh.offsets(p)
        self.lsize = self.mesh.lsize(self.pl)
        self.lsize_fine = self.mesh.lsize(p)
        self.B, self.D, _, self.qw = oracle.basis_1d(self.P, self.Q, 0)
        self.Bf, self.Df, _, _ = oracle.basis_1d(self.Pf, self.Q, 0)
        self.xoffsets = self.mesh.offsets(1)
        self.xcoord = self.mesh.coord_lvector()
        self.qdata = oracle.setup_geo(self.nelem, self.Q, self.xoffsets, self.xcoord, which)
        self.has_gradu = oracle.PROBLEMS[problem][2]
        self.gradu = np.zeros((self.nelem, 9, self.Q ** 3)) if self.has_gradu else None
        # state on the FINE level (gradu is always produced by the fine residual operator)
        self.u_fine = smooth_displacement(self.mesh.node_coords(p), scale).reshape(-1)
        self.residual_fine(self.u_fine)

    def to_perm(self, v_lex):
        """Re-order a lexicographic level L-vector into the (optionally permuted) numbering."""
        if self.perm is None:
            return v_lex
        out = np.empty_like(v_lex).reshape(-1, 3)
        out[self.perm] = v_lex.reshape(-1, 3)
        return out.reshape(-1)

    def residual_fine(self, u):
        """Residual operator on the fine level (writes gradu as a side effect)."""
        return oracle.operator_apply(self.problem, False, PHYS, self.nelem, self.Pf, self.Q, self.Bf,
                                     self.Df, self.offsets_fine, self.qdata, self.gradu, u, self.which)

    def jacobian(self, x):
        return oracle.operator_apply(self.problem, True, PHYS, self.nelem, self.P, self.Q, self.B, self.D,
                                     self.offsets, self.qdata, self.gradu, x, self.which)

    def diagonal(self):
        return oracle.operator_diagonal(self.problem, PHYS, self.nelem, self.P, self.Q, self.B, self.D,
                                        self.offsets, self.qdata, self.gradu, self.lsize, self.which)


def cube_rotations():
    """The 24 proper rotations of the reference cube as (perm, flip): local axis d of a rotated element runs along
    old local axis perm[d], reversed where flip[d].  Reflections are left out: they would turn detJ negative."""
    import itertools
    out = []
    for perm in itertools.permutations(range(3)):
        sign = np.linalg.det(np.eye(3)[list(perm)])
        for flip in itertools.product((0, 1), repeat=3):
            if sign * (-1) ** sum(flip) > 0:
                out.append((perm, flip))
    assert len(out) == 24
    return out


def reoriented(mesh, seed=0):
    """exodus.HexMesh with the elements of `mesh` (a HexMesh, or anything with vertices and offsets(1) such as a
    BoxMesh), each re-listed under a seeded random one of the 24 cube rotations: the same conforming mesh, but
    neighbouring elements no longer share their local axes.  Side sets are renumbered to the rotated local faces."""
    from ceedpetscsolid_b200.exodus import _SIDE, HexMesh
    coords = np.asarray(mesh.vertices, dtype=np.float64).reshape(-1, 3)
    conn = np.asarray(mesh.connect if hasattr(mesh, "connect") else mesh.offsets(1) // 3, dtype=np.int64)
    rots = cube_rotations()
    pick = np.random.default_rng(seed).integers(0, 24, conn.shape[0])
    # tensor vertex t' = i' + 2 j' + 4 k' of the rotated element is old vertex t with v[perm[d]] = v'[d] ^ flip[d]
    tables = []
    for perm, flip in rots:
        tab = np.empty(8, dtype=np.int64)
        for t2 in range(8):
            v2 = [(t2 >> d) & 1 for d in range(3)]
            v = [0, 0, 0]
            for d in range(3):
                v[perm[d]] = v2[d] ^ flip[d]
            tab[t2] = v[0] + 2 * v[1] + 4 * v[2]
        tables.append(tab)
    new = np.stack([conn[e, tables[r]] for e, r in enumerate(pick)])
    sidesets = {}
    face = {s: [t for t in range(8) if ((t >> ax) & 1) == side] for s, (ax, side) in _SIDE.items()}
    for sid, (els, sides) in getattr(mesh, "sidesets", {}).items():
        ns = []
        for e, s in zip(np.asarray(els), np.asarray(sides)):
            target = set(conn[e, face[int(s)]])
            ns.append(next(s2 for s2 in face if set(new[e, face[s2]]) == target))
        sidesets[sid] = (np.asarray(els), np.asarray(ns, dtype=np.int64))
    return HexMesh(coords, new, sidesets)


def rel_err(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / max(np.linalg.norm(np.asarray(b)), 1e-300)


def lattice_ids(N):
    """(i, j, k) of every node of an (Nx, Ny, Nz) node lattice, x fastest"""
    k, j, i = np.meshgrid(np.arange(N[2]), np.arange(N[1]), np.arange(N[0]), indexing="ij")
    return i.reshape(-1), j.reshape(-1), k.reshape(-1)


def dense_from_stencil(sv, N):
    """Dense matrix of a 27-point block stencil in the layout of b200_stencil27_spmv,
    sv[((dx+1) + 3(dy+1) + 9(dz+1))*3 + b][row]; entries that point outside the lattice are not read."""
    n = 3 * int(np.prod(N))
    i, j, k = lattice_ids(N)
    A = np.zeros((n, n))
    for o in range(27):
        dx, dy, dz = o % 3 - 1, (o // 3) % 3 - 1, o // 9 - 1
        ok = (i + dx >= 0) & (i + dx < N[0]) & (j + dy >= 0) & (j + dy < N[1]) & (k + dz >= 0) & (k + dz < N[2])
        colnode = (i + dx) + N[0] * ((j + dy) + N[1] * (k + dz))
        for a in range(3):
            for b in range(3):
                r = np.flatnonzero(ok) * 3 + a
                A[r, colnode[ok] * 3 + b] = sv[o * 3 + b, r]
    return A
