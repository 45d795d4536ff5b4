"""Structured hex box meshes: the DMPlex stand-in used by the harness.

The reference obtains its mesh, the tensor-ordered cell closures and the local/global
dof numbering from PETSc DMPlex (`CreateDistributedDM` /root/reference/src/setupdm.c:40-68,
`SetupDMByDegree` :138-201, `CreateRestrictionPlex` /root/reference/src/setuplibceed.c:194-240).
PETSc is not available here, so this module produces the same *inputs to libCEED* for
`-dm_plex_box_faces nx,ny,nz` boxes:

* `offsets[nelem][P^3]` : L-vector index of component 0 of every element node, x fastest
  (what `CreateRestrictionPlex` passes to `CeedElemRestrictionCreate` with compstride 1);
* interlaced `[node][3]` L-vectors that include Dirichlet nodes (and ghosts, when partitioned);
* vertex coordinates + a P=2 coordinate restriction (`Erestrictx`, setuplibceed.c:279-280);
* the Dirichlet mask (`-test` marks every boundary face, setupdm.c:160-170).

A brick partition (`partition`) provides the owned/ghost split that `DMPlexDistribute`
(overlap 0, setupdm.c:58-64) would give, for the multi-GPU halo exchange.
"""
from dataclasses import dataclass, field

import numpy as np


def gll_nodes(P):
    """Gauss-Lobatto-Legendre nodes on [-1,1] (host-side, Newton on P'_{P-1})."""
    n = P - 1
    if P == 2:
        return np.array([-1.0, 1.0])
    x = -np.cos(np.pi * np.arange(P) / n)
    for _ in range(100):
        p0, p1 = np.ones_like(x), x.copy()
        for j in range(2, n + 1):
            p0, p1 = p1, ((2 * j - 1) * x * p1 - (j - 1) * p0) / j
        with np.errstate(divide="ignore", invalid="ignore"):
            dp = n * (x * p1 - p0) / (x * x - 1)
            d2p = (2 * x * dp - n * (n + 1) * p1) / (1 - x * x)
            dx = dp / d2p
        dx[0] = dx[-1] = 0.0
        x = x - dx
        if np.max(np.abs(dx)) < 1e-16:
            break
    x[0], x[-1] = -1.0, 1.0
    return x


@dataclass
class BoxMesh:
    """Box [0,lx]x[0,ly]x[0,lz] with n=(nx,ny,nz) hexes, or a brick sub-range of it.

    `origin`/`gn` describe a brick of a larger global box (for partitioned runs):
    this mesh holds elements [origin, origin+n) of the global `gn` box.
    """
    n: tuple
    perturb: float = 0.0
    seed: int = 0
    lengths: tuple = (1.0, 1.0, 1.0)
    origin: tuple = (0, 0, 0)
    gn: tuple = None
    vertices: np.ndarray = field(default=None, repr=False)
    # element numbering: row i of offsets() is lexicographic element elem_order[i] (None = lexicographic).
    # brick(..., interface_first=True) puts the elements that touch a partition interface first
    # (n_interface of them, padded to a multiple of 16) so that their part of an operator application can run,
    # and the halo exchange start, before the interior elements are processed.
    elem_order: np.ndarray = field(default=None, repr=False)
    n_interface: int = 0

    def __post_init__(self):
        self.n = tuple(int(v) for v in self.n)
        if self.gn is None:
            self.gn = self.n
        self.gn = tuple(int(v) for v in self.gn)
        self.nelem = self.n[0] * self.n[1] * self.n[2]
        if self.vertices is None:
            self.vertices = self._make_vertices()

    # ---------------------------------------------------------------- geometry
    def _make_vertices(self):
        """(nvz, nvy, nvx, 3) vertex coordinates of this brick.  The perturbation of the
        GLOBAL box is generated (seeded) and sliced so that bricks agree on shared vertices."""
        gnx, gny, gnz = self.gn
        ax = [np.linspace(0.0, self.lengths[d], self.gn[d] + 1) for d in range(3)]
        Z, Y, X = np.meshgrid(ax[2], ax[1], ax[0], indexing="ij")
        V = np.stack([X, Y, Z], axis=-1)
        if self.perturb:
            rng = np.random.default_rng(self.seed)
            h = min(self.lengths[d] / self.gn[d] for d in range(3))
            d = self.perturb * h * (rng.random(V.shape) - 0.5)
            d[0, :, :, :] = 0; d[-1, :, :, :] = 0
            d[:, 0, :, :] = 0; d[:, -1, :, :] = 0
            d[:, :, 0, :] = 0; d[:, :, -1, :] = 0
            V = V + d
        ox, oy, oz = self.origin
        nx, ny, nz = self.n
        return np.ascontiguousarray(V[oz:oz + nz + 1, oy:oy + ny + 1, ox:ox + nx + 1])

    def coord_lvector(self):
        """Interlaced vertex-coordinate L-vector (what DMGetCoordinatesLocal gives)."""
        return np.ascontiguousarray(self.vertices.reshape(-1, 3)).reshape(-1)

    # ---------------------------------------------------------------- numbering
    def nodes_per_dim(self, p):
        return tuple(self.n[d] * p + 1 for d in range(3))

    def num_nodes(self, p):
        N = self.nodes_per_dim(p)
        return N[0] * N[1] * N[2]

    def lsize(self, p, ncomp=3):
        return ncomp * self.num_nodes(p)

    def offsets(self, p, ncomp=3, node_perm=None):
        """int32 [nelem, (p+1)^3]: dof index of component 0, tensor (x fastest) closure order."""
        P = p + 1
        nx, ny, nz = self.n
        Nx, Ny, Nz = self.nodes_per_dim(p)
        ez, ey, ex = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
        base = (ex * p + Nx * (ey * p + Ny * (ez * p))).reshape(-1, 1)
        c, b, a = np.meshgrid(np.arange(P), np.arange(P), np.arange(P), indexing="ij")
        loc = (a + Nx * (b + Ny * c)).reshape(1, -1)
        nodes = base + loc
        if self.elem_order is not None:
            nodes = nodes[self.elem_order]
        if node_perm is not None:
            nodes = node_perm[nodes]
        off = nodes * ncomp
        assert off.max() < 2 ** 31
        return np.ascontiguousarray(off.astype(np.int32))

    @property
    def elem_ids(self):
        """global element ids (lexicographic in the `gn` box) of the rows of offsets()"""
        ez, ey, ex = np.meshgrid(*(np.arange(self.n[d]) + self.origin[d] for d in (2, 1, 0)), indexing="ij")
        ids = (ex + self.gn[0] * (ey + self.gn[1] * ez)).reshape(-1).astype(np.int64)
        return ids if self.elem_order is None else ids[self.elem_order]

    def node_coords(self, p):
        """(num_nodes, 3) physical coordinates of the degree-p GLL nodes (trilinear geometry)."""
        P = p + 1
        nx, ny, nz = self.n
        Nx, Ny, Nz = self.nodes_per_dim(p)
        r = (gll_nodes(P) + 1) / 2
        V = self.vertices
        out = np.zeros((Nz, Ny, Nx, 3))
        w0, w1 = 1 - r, r
        for c in range(P):
            for b in range(P):
                for a in range(P):
                    val = 0
                    for dz, wz in ((0, w0[c]), (1, w1[c])):
                        for dy, wy in ((0, w0[b]), (1, w1[b])):
                            for dx, wx in ((0, w0[a]), (1, w1[a])):
                                val = val + wz * wy * wx * V[dz:dz + nz, dy:dy + ny, dx:dx + nx]
                    out[c:c + nz * p:p, b:b + ny * p:p, a:a + nx * p:p] = val
        return out.reshape(-1, 3)

    def boundary_mask(self, p, faces="all"):
        """bool [num_nodes]: nodes on the selected faces of the GLOBAL box.
        faces: "all" (the `-test` marker label) or an iterable of (axis, side) with side in {0,1}."""
        Nx, Ny, Nz = self.nodes_per_dim(p)
        m = np.zeros((Nz, Ny, Nx), dtype=bool)
        if faces == "all":
            faces = [(a, s) for a in range(3) for s in (0, 1)]
        for axis, side in faces:
            at_global = (self.origin[axis] == 0) if side == 0 else (
                self.origin[axis] + self.n[axis] == self.gn[axis])
            if not at_global:
                continue
            idx = [slice(None)] * 3
            idx[2 - axis] = 0 if side == 0 else -1
            m[tuple(idx)] = True
        return m.reshape(-1)

    # ---------------------------------------------------------------- partition
    def brick(self, grid, rank, interface_first=False):
        """Sub-mesh of rank `rank` in a `grid=(px,py,pz)` brick partition (x fastest)."""
        px, py, pz = grid
        rx, ry, rz = rank % px, (rank // px) % py, rank // (px * py)
        lo, sz = [], []
        for d, (pp, rr) in enumerate(((px, rx), (py, ry), (pz, rz))):
            q, rem = divmod(self.n[d], pp)
            start = rr * q + min(rr, rem)
            lo.append(self.origin[d] + start)
            sz.append(q + (1 if rr < rem else 0))
        order, nif = None, 0
        if interface_first:
            ez, ey, ex = np.meshgrid(np.arange(sz[2]), np.arange(sz[1]), np.arange(sz[0]), indexing="ij")
            touch = np.zeros(ex.shape, bool)
            for d, (e, pp, rr) in enumerate(((ex, px, rx), (ey, py, ry), (ez, pz, rz))):
                if rr > 0:
                    touch |= e == 0
                if rr < pp - 1:
                    touch |= e == sz[d] - 1
            touch = touch.reshape(-1)
            order = np.concatenate([np.flatnonzero(touch), np.flatnonzero(~touch)])  # stable: lexicographic inside each part
            nif = int(touch.sum())
            nif = min(order.size, (nif + 15) // 16 * 16) if nif else 0
        return BoxMesh(n=tuple(sz), perturb=self.perturb, seed=self.seed, lengths=self.lengths,
                       origin=tuple(lo), gn=self.gn, elem_order=order, n_interface=nif)


def smooth_displacement(X, scale=0.02):
    """Admissible smooth state of SURVEY.md 8(d): u = s*(sin2x*cosy+z^2, xy-z/2, e^{z/2}x-y^2)."""
    x, y, z = X[:, 0], X[:, 1], X[:, 2]
    return scale * np.stack([np.sin(2 * x) * np.cos(y) + z * z, x * y - z / 2,
                             np.exp(z / 2) * x - y * y], axis=-1)


def grid_for(nranks):
    """Brick grids used for 1/2/4/8 GPUs (SURVEY.md 8(e))."""
    return {1: (1, 1, 1), 2: (2, 1, 1), 4: (2, 2, 1), 8: (2, 2, 2)}[nranks]
