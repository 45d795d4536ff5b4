"""Unstructured hex8 meshes (`-mesh file.exo`): the DMPlexCreateFromFile branch of
/root/reference/src/setupdm.c:40-68 for the meshes the reference ships (meshes/Tube8_*_2ss_us.exo: one HEX8 block,
two side sets that `-bc_clamp 1,2` refers to).

* `read_exodus` / `write_exodus`: the subset of Exodus II (NetCDF-3 classic, via scipy.io) those files use.
* `HexMesh`: the same interface as `mesh.BoxMesh` (offsets, node coordinates, Dirichlet masks) for an arbitrary
  conforming hex8 mesh with trilinear geometry.  Degree-p nodes are numbered TOPOLOGICALLY: a node is identified by
  the set of (vertex id, integer trilinear weight) pairs with non-zero weight, which is the same for every element
  sharing the vertex / edge / face it lies on (GLL points are symmetric, so edge and face orientations cannot
  disagree) -- no coordinate hashing, no tolerance.
* `HexMesh.brick` / `HexSubMesh`: one part of a recursive coordinate bisection of the elements, for partitioned runs
  (the DMPlexDistribute step of setupdm.c:58-64); halo.Halo builds the shared-node sets from the parts' node ids.
* `tube_mesh`: a synthetic quarter/half/full tube of hexes with the two end faces as side sets 1 and 2, used by the
  tests (the reference's own files are read where /root/reference is mounted, never copied).
"""
import numpy as np

from .mesh import gll_nodes

# Exodus HEX8 node order -> tensor order t = i + 2 j + 4 k (x fastest)
_EXO_TO_TENSOR = np.array([0, 1, 3, 2, 4, 5, 7, 6])
# Exodus HEX8 side number (1-based) -> (axis, side) in tensor coordinates
_SIDE = {1: (1, 0), 2: (0, 1), 3: (1, 1), 4: (0, 0), 5: (2, 0), 6: (2, 1)}


def read_exodus(path):
    """-> dict(coords (N,3) float64, connect (E,8) int64 zero-based in TENSOR order, sidesets {id: (elems, sides)})."""
    from scipy.io import netcdf_file
    nc = netcdf_file(path, "r", mmap=False)
    v = nc.variables
    if "coord" in v:
        coords = np.array(v["coord"].data, dtype=np.float64).T
    else:
        coords = np.stack([np.array(v[k].data, dtype=np.float64) for k in ("coordx", "coordy", "coordz")], axis=1)
    nblk = nc.dimensions.get("num_el_blk", 1)
    blocks = []
    for b in range(1, nblk + 1):
        c = v[f"connect{b}"]
        et = getattr(c, "elem_type", b"HEX8")
        et = et.decode() if isinstance(et, bytes) else str(et)
        if not et.upper().startswith("HEX") or c.data.shape[1] != 8:
            raise ValueError(f"{path}: element block {b} is {et} with {c.data.shape[1]} nodes; only HEX8 is supported")
        blocks.append(np.array(c.data, dtype=np.int64) - 1)
    connect = np.concatenate(blocks)[:, _tensor_from_exo()]
    ids = np.array(v["ss_prop1"].data, dtype=np.int64) if "ss_prop1" in v else np.arange(1, nc.dimensions.get("num_side_sets", 0) + 1)
    sidesets = {}
    for s, sid in enumerate(ids, start=1):
        sidesets[int(sid)] = (np.array(v[f"elem_ss{s}"].data, dtype=np.int64) - 1, np.array(v[f"side_ss{s}"].data, dtype=np.int64))
    nc.close()
    return dict(coords=coords, connect=connect, sidesets=sidesets)


def _tensor_from_exo():
    """column permutation: tensor-ordered connectivity[:, t] = exodus connectivity[:, perm[t]]"""
    perm = np.empty(8, dtype=np.int64)
    perm[_EXO_TO_TENSOR] = np.arange(8)
    return perm


def write_exodus(path, coords, connect_tensor, sidesets):
    """Minimal Exodus II writer (one HEX8 block + side sets), the counterpart of read_exodus."""
    from scipy.io import netcdf_file
    E, N = connect_tensor.shape[0], coords.shape[0]
    nc = netcdf_file(path, "w", version=2)
    for k, n in (("num_dim", 3), ("num_nodes", N), ("num_elem", E), ("num_el_blk", 1), ("num_el_in_blk1", E),
                 ("num_nod_per_el1", 8), ("num_side_sets", len(sidesets)), ("len_string", 33)):
        nc.createDimension(k, n)
    for a, k in enumerate(("coordx", "coordy", "coordz")):
        var = nc.createVariable(k, "d", ("num_nodes",))
        var[:] = coords[:, a]
    exo = np.empty_like(connect_tensor)
    exo[:, np.arange(8)] = connect_tensor[:, _EXO_TO_TENSOR]   # exodus column e holds tensor column _EXO_TO_TENSOR[e]
    c = nc.createVariable("connect1", "i", ("num_el_in_blk1", "num_nod_per_el1"))
    c[:] = exo + 1
    c.elem_type = b"HEX8"
    if sidesets:
        p = nc.createVariable("ss_prop1", "i", ("num_side_sets",))
        p[:] = np.array(sorted(sidesets), dtype=np.int32)
        for s, sid in enumerate(sorted(sidesets), start=1):
            el, sd = sidesets[sid]
            nc.createDimension(f"num_side_ss{s}", len(el))
            ve = nc.createVariable(f"elem_ss{s}", "i", (f"num_side_ss{s}",))
            ve[:] = np.asarray(el) + 1
            vs = nc.createVariable(f"side_ss{s}", "i", (f"num_side_ss{s}",))
            vs[:] = np.asarray(sd)
    nc.close()


class HexMesh:
    """Conforming hex8 mesh, trilinear geometry; same interface as mesh.BoxMesh (brick() gives a part of it for
    partitioned runs)."""
    structured = False
    elem_order = None
    n_interface = 0

    def __init__(self, coords, connect, sidesets=None):
        self.vertices = np.ascontiguousarray(coords, dtype=np.float64)        # (Nv, 3)
        self.connect = np.ascontiguousarray(connect, dtype=np.int64)          # (E, 8) tensor order
        self.sidesets = dict(sidesets or {})
        self.nelem = self.connect.shape[0]
        self._cache = {}

    @classmethod
    def from_file(cls, path):
        d = read_exodus(path)
        return cls(d["coords"], d["connect"], d["sidesets"])

    # ---------------------------------------------------------------- numbering
    def _level(self, p):
        """(elem_nodes (E, P^3) node ids in tensor order, num_nodes) of the degree-p discretisation"""
        if p in self._cache:
            return self._cache[p]
        P, E = p + 1, self.nelem
        if p == 1:
            out = (self.connect.copy(), self.vertices.shape[0])
            self._cache[p] = out
            return out
        a = np.arange(P)
        w1 = np.stack([p - a, a], axis=1)                                     # integer 1-D weights of the two ends
        # weight of vertex (i,j,k) at lattice node (a,b,c): w1[a,i] w1[b,j] w1[c,k]; node index a + P(b + P c)
        W = np.einsum("ai,bj,ck->cbakji", w1, w1, w1).reshape(P ** 3, 8)     # columns in tensor vertex order
        vid = np.broadcast_to(self.connect[:, None, :], (E, P ** 3, 8))
        wgt = np.broadcast_to(W[None], (E, P ** 3, 8))
        vid = np.where(wgt > 0, vid, -1)
        order = np.argsort(vid, axis=2, kind="stable")
        key = np.concatenate([np.take_along_axis(vid, order, 2), np.take_along_axis(wgt * (vid >= 0), order, 2)], axis=2)
        _, inv = np.unique(key.reshape(E * P ** 3, 16), axis=0, return_inverse=True)
        ids = inv.reshape(E, P ** 3).astype(np.int64)
        out = (ids, int(ids.max()) + 1)
        self._cache[p] = out
        return out

    def num_nodes(self, p):
        return self._level(p)[1]

    def lsize(self, p, ncomp=3):
        return ncomp * self.num_nodes(p)

    def offsets(self, p, ncomp=3, node_perm=None):
        ids = self._level(p)[0]
        if node_perm is not None:
            ids = node_perm[ids]
        off = ids * ncomp
        assert off.max() < 2 ** 31
        return np.ascontiguousarray(off.astype(np.int32))

    def coord_lvector(self):
        return self.vertices.reshape(-1).copy()

    def node_coords(self, p):
        """(num_nodes, 3) physical coordinates of the degree-p GLL nodes (trilinear map of the reference nodes)."""
        P = p + 1
        ids, nn = self._level(p)
        r = (gll_nodes(P) + 1) / 2
        w1 = np.stack([1 - r, r], axis=1)
        W = np.einsum("ai,bj,ck->cbakji", w1, w1, w1).reshape(P ** 3, 8)
        xe = np.einsum("nv,evd->end", W, self.vertices[self.connect])        # (E, P^3, 3)
        out = np.zeros((nn, 3))
        out[ids.reshape(-1)] = xe.reshape(-1, 3)
        return out

    # ---------------------------------------------------------------- boundary
    def _side_nodes(self, p, axis, side):
        """lattice indices (within an element) of the P^2 nodes on tensor side (axis, side)"""
        P = p + 1
        c, b, a = np.meshgrid(np.arange(P), np.arange(P), np.arange(P), indexing="ij")
        sel = (a, b, c)[axis] == (0 if side == 0 else p)
        return np.flatnonzero(sel.reshape(-1))

    def boundary_faces(self):
        """(elems, exodus side numbers) of all faces that belong to one element only"""
        face_vertices = {s: self._side_nodes(1, *_SIDE[s]) for s in _SIDE}
        keys, owner = [], []
        for s, loc in face_vertices.items():
            fv = np.sort(self.connect[:, loc], axis=1)
            keys.append(fv)
            owner.append(np.stack([np.arange(self.nelem), np.full(self.nelem, s)], axis=1))
        keys, owner = np.concatenate(keys), np.concatenate(owner)
        _, inv, cnt = np.unique(keys, axis=0, return_inverse=True, return_counts=True)
        ext = cnt[inv] == 1
        return owner[ext, 0], owner[ext, 1]

    def boundary_mask(self, p, faces="all"):
        """bool [num_nodes]: nodes on the selected side sets (ids as in the file) or on the whole boundary ("all")."""
        ids, nn = self._level(p)
        m = np.zeros(nn, dtype=bool)
        if faces == "all":
            sets = [self.boundary_faces()]
        else:
            sets = [self.sidesets[int(f)] for f in faces]
        for el, sd in sets:
            for s in np.unique(sd):
                loc = self._side_nodes(p, *_SIDE[int(s)])
                m[ids[np.asarray(el)[sd == s]][:, loc].reshape(-1)] = True
        return m

    # ---------------------------------------------------------------- partition
    def partition(self, nparts):
        """list of nparts ascending global element-id arrays: recursive coordinate bisection of the element centroids.
        Each step splits the longest centroid extent of the current set into nparts//2 and nparts - nparts//2 parts with
        element counts in proportion; the sort is stable with the element id as tie-break, so every rank computes the
        same partition without communication."""
        key = ("parts", nparts)
        if key in self._cache:
            return self._cache[key]
        cen = self.vertices[self.connect].mean(axis=1)
        parts = []

        def split(ids, k):
            if k == 1:
                parts.append(np.sort(ids))
                return
            c = cen[ids]
            axis = int(np.argmax(c.max(axis=0) - c.min(axis=0))) if ids.size else 0
            ids = ids[np.lexsort((ids, c[:, axis]))]
            k1 = k // 2
            n1 = ids.size * k1 // k
            split(ids[:n1], k1)
            split(ids[n1:], k - k1)

        split(np.arange(self.nelem, dtype=np.int64), int(nparts))
        empty = [r for r, p in enumerate(parts) if p.size == 0]
        if empty:
            raise ValueError(f"partition of {self.nelem} elements into {nparts} parts leaves part(s) {empty} empty")
        self._cache[key] = parts
        return parts

    def part_node_ids(self, nparts, p):
        """per part: ascending global ids of the degree-p nodes it holds"""
        key = ("part_nodes", nparts, p)
        if key not in self._cache:
            ids = self._level(p)[0]
            self._cache[key] = [np.unique(ids[e]) for e in self.partition(nparts)]
        return self._cache[key]

    def brick(self, grid, rank, interface_first=False):
        """Part `rank` of a prod(grid)-way partition (HexMesh.partition) as a HexSubMesh, the counterpart of
        BoxMesh.brick.  interface_first: the elements with a vertex held by another part come first (n_interface of
        them, padded to a multiple of 16), so that an operator application can start the halo exchange before the
        interior elements; a vertex held by another part is a superset of a shared dof at every degree."""
        k = int(np.prod(grid))
        elems = self.partition(k)[rank]
        order, nif = None, 0
        if interface_first:
            held = np.zeros(self.vertices.shape[0], dtype=np.int64)
            for v in self.part_node_ids(k, 1):
                held[v] += 1
            touch = (held[self.connect[elems]] > 1).any(axis=1)
            order = np.concatenate([np.flatnonzero(touch), np.flatnonzero(~touch)])
            nif = int(touch.sum())
            nif = min(order.size, (nif + 15) // 16 * 16) if nif else 0
        return HexSubMesh(self, elems if order is None else elems[order], order, nif)


class HexSubMesh:
    """One part of a partitioned HexMesh, with the HexMesh interface the DM and set-up code use.  Local node ids of
    every degree run over the part's nodes in ascending global (parent topological) id; `elem_ids` are the global ids
    of the rows of offsets(); row i is the part's element elem_order[i] in ascending-id order (None: that order).
    Dirichlet masks and node coordinates are the parent's, restricted to the part, so a node on a clamped side set
    is masked on every part that holds it, also where the part touches the node through an edge only."""
    structured = False

    def __init__(self, parent, elem_ids, elem_order, n_interface):
        self.parent, self.elem_ids = parent, np.asarray(elem_ids, dtype=np.int64)
        self.elem_order, self.n_interface = elem_order, int(n_interface)
        self.nelem = self.elem_ids.size
        self._cache = {}
        self.vertices = parent.vertices[self.node_ids(1)]

    def _level(self, p):
        if p not in self._cache:
            gids = self.parent._level(p)[0][self.elem_ids]
            nodes = np.unique(gids)
            self._cache[p] = (np.searchsorted(nodes, gids), nodes)
        return self._cache[p]

    def node_ids(self, p):
        """ascending global ids of the local degree-p nodes (local -> global)"""
        return self._level(p)[1]

    def num_nodes(self, p):
        return self.node_ids(p).size

    def lsize(self, p, ncomp=3):
        return ncomp * self.num_nodes(p)

    def offsets(self, p, ncomp=3, node_perm=None):
        ids = self._level(p)[0]
        if node_perm is not None:
            ids = node_perm[ids]
        off = ids * ncomp
        assert off.max() < 2 ** 31
        return np.ascontiguousarray(off.astype(np.int32))

    def coord_lvector(self):
        return self.vertices.reshape(-1).copy()

    def node_coords(self, p):
        return self.parent.node_coords(p)[self.node_ids(p)]

    def boundary_mask(self, p, faces="all"):
        return self.parent.boundary_mask(p, faces)[self.node_ids(p)]


def tube_mesh(nr=2, nt=8, nz=4, r0=0.5, r1=1.0, length=2.0, angle=2 * np.pi):
    """Synthetic tube (annulus x length) of nr x nt x nz hexes; side set 1 = face z = 0, side set 2 = face z = length.
    angle < 2 pi gives an open sector; the full tube is periodic in the angle (shared vertices)."""
    closed = abs(angle - 2 * np.pi) < 1e-12
    nth = nt if closed else nt + 1
    rr = np.linspace(r0, r1, nr + 1)
    th = np.linspace(0.0, angle, nt + 1)[:nth]
    zz = np.linspace(0.0, length, nz + 1)
    K, T, R = np.meshgrid(np.arange(nz + 1), np.arange(nth), np.arange(nr + 1), indexing="ij")
    coords = np.stack([rr[R] * np.cos(th[T]), rr[R] * np.sin(th[T]), zz[K]], axis=-1).reshape(-1, 3)
    vid = lambda i, j, k: (i) + (nr + 1) * ((j % nth) + nth * k)
    conn, ss1, ss2 = [], ([], []), ([], [])
    for k in range(nz):
        for j in range(nt):
            for i in range(nr):
                e = len(conn)
                # tensor axes: x = radial, y = angular, z = axial (right-handed: r x theta = z)
                conn.append([vid(i + di, j + dj, k + dk) for dk in (0, 1) for dj in (0, 1) for di in (0, 1)])
                if k == 0:
                    ss1[0].append(e); ss1[1].append(5)
                if k == nz - 1:
                    ss2[0].append(e); ss2[1].append(6)
    sidesets = {1: (np.array(ss1[0]), np.array(ss1[1])), 2: (np.array(ss2[0]), np.array(ss2[1]))}
    return HexMesh(coords, np.array(conn, dtype=np.int64), sidesets)
