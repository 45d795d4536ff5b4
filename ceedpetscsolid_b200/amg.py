"""Smoothed-aggregation algebraic multigrid on the assembled p = 1 level: the GAMG coarse solve of the reference
(`preonly` + GAMG, /root/reference/elasticity.c:569-585) for meshes without a node lattice (-mesh file.exo), where the
geometric h-multigrid (solver.HMultigrid) cannot coarsen.

Set-up is split in two:

* symbolic, once per mesh, on the host (numpy): node graph of the p = 1 level, deterministic greedy aggregation,
  tentative prolongator from the six rigid-body modes of every aggregate (thin QR; R is the next level's near-null
  space), and the block patterns of A P_tent, P = (I - omega D^-1 A) P_tent, P^T and A_c = P^T A P.  Every output
  block of a product gets its pair list: the (A block, B block) index pairs that contribute to it, in a fixed order.
  GAMG's default threshold of 0 keeps every edge, so the aggregates depend on the mesh graph alone.
* numeric, once per Newton step, on the device: level-0 BSR values from the CeedOperatorLinearAssemble element
  matrices, lambda_max(D^-1 A), the pair-list products and the transposed prolongator by a fixed gather
  (csrc/b200_amg.cu: no atomics, bit-identical from run to run), and a dense Cholesky factor of the coarsest level.

The coarse solve is one V(2,2) cycle with Chebyshev/Jacobi smoothing and an exact coarsest solve: a fixed symmetric
linear operator, as HMultigrid.solve, with no host synchronisation.  On CPU tensors (oracle runs) every kernel has a
torch branch with the same arithmetic.
"""
import time
import warnings

import numpy as np
import torch

from .ceed import b2, lib
from . import solver

MAX_COARSE_DOFS = 1500    # the coarsest level is solved directly once it has at most this many rows
MIN_AGGREGATE = 3         # smaller aggregates are merged into a neighbour
MIN_SHRINK = 4.0          # coarsening stops when a level shrinks by less than this factor
MAX_LEVELS = 10
MAX_DENSE_COARSEST = 16000   # rows: the coarsest level is factored densely (two n^2 FP64 matrices: 4 GB at this size)


# --------------------------------------------------------------------------- symbolic set-up (host)


def node_graph(elem_nodes, nn):
    """CSR (indptr, indices) of the node graph: two nodes are adjacent if they share an element (diagonal included),
    column indices sorted in every row."""
    en = np.asarray(elem_nodes, dtype=np.int64)
    k = en.shape[1]
    key = np.unique((np.repeat(en, k, axis=1) * nn + np.tile(en, (1, k))).reshape(-1))
    rows = key // nn
    return np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=nn))]).astype(np.int64), key % nn


def aggregate(indptr, indices, free, min_size=MIN_AGGREGATE):
    """Greedy distance-1 aggregation in node order (Vanek-style), on the graph restricted to the free nodes:
      1. a node whose whole free neighbourhood is unaggregated becomes a root: it and its neighbours form an aggregate;
      2. a leftover node joins the first (lowest-numbered) neighbour's aggregate of step 1;
      3. what is still left forms aggregates with its unaggregated neighbours, in node order;
      4. aggregates with fewer than `min_size` nodes are merged into the aggregate of their first neighbour outside.
    Returns (agg [n] aggregate id, -1 for constrained nodes; number of aggregates).  Deterministic."""
    n = free.size
    agg = np.full(n, -1, dtype=np.int64)
    nbrs = [None] * n

    def nb(i):
        if nbrs[i] is None:
            v = indices[indptr[i]:indptr[i + 1]]
            nbrs[i] = v[free[v]]
        return nbrs[i]

    na = 0
    for i in range(n):
        if free[i] and agg[i] < 0:
            v = nb(i)
            if (agg[v] < 0).all():
                agg[v] = na
                agg[i] = na
                na += 1
    phase1 = agg.copy()
    for i in np.flatnonzero(free & (agg < 0)):
        a = phase1[nb(i)]
        a = a[a >= 0]
        if a.size:
            agg[i] = a[0]
    for i in np.flatnonzero(free & (agg < 0)):
        if agg[i] < 0:
            v = nb(i)
            v = v[agg[v] < 0]
            agg[v] = na
            agg[i] = na
            na += 1
    sizes = np.bincount(agg[agg >= 0], minlength=na)
    for a in np.flatnonzero((sizes > 0) & (sizes < min_size)):
        if sizes[a] == 0 or sizes[a] >= min_size:
            continue
        members = np.flatnonzero(agg == a)
        target = -1
        for i in members:
            o = agg[nb(i)]
            o = o[(o >= 0) & (o != a)]
            if o.size:
                target = o[0]
                break
        if target >= 0:
            agg[members] = target
            sizes[target] += sizes[a]
            sizes[a] = 0
    used = np.unique(agg[agg >= 0])
    out = np.full(n, -1, dtype=np.int64)
    out[agg >= 0] = np.searchsorted(used, agg[agg >= 0])
    return out, used.size


def _rotations(d):
    """(..., 3, 3): column k = displacement at offset d under a unit rotation about axis k (x, y, z)"""
    W = np.zeros(d.shape[:-1] + (3, 3))
    W[..., 1, 0], W[..., 2, 0] = -d[..., 2], d[..., 1]
    W[..., 0, 1], W[..., 2, 1] = d[..., 2], -d[..., 0]
    W[..., 0, 2], W[..., 1, 2] = -d[..., 1], d[..., 0]
    return W


def rigid_body_modes(coords, center):
    """(n, 3, 6) near-null space of elasticity per node: three translations and three rotations about ONE common point
    `center` -- the same six global modes at every node, so that a coarse coefficient vector shared by neighbouring
    aggregates still describes one rigid motion."""
    B = np.zeros((coords.shape[0], 3, 6))
    B[:, :, :3] = np.eye(3)
    B[:, :, 3:] = _rotations(coords - center)
    return B


def tentative_prolongator(agg, nagg, B, xyz, weight, center, level=0, tol=1e-12):
    """Per aggregate: the stacked near-null blocks of its nodes (b n_a x 6), thin QR with a non-negative diagonal of R.
    B holds the global rigid-body modes about `center` (level 0: rigid_body_modes; below: the R of the level above);
    xyz, weight: node positions and weights (level 0: coordinates and 1; below: aggregate centroids and node counts).
    For conditioning the QR is taken of the modes re-centred on the aggregate's centroid c_a, B S_a^-1 = Q R with
    S_a = [[I, W(c_a - center)], [0, I]] (an exact change of basis), and the next level's near-null block is R S_a: the
    coarse vector e_k on every aggregate is the same global mode k on every level.
    Returns (Q values [n_free, b, 6] in node order, R S [nagg, 6, 6], centroids [nagg, 3], weights [nagg]).  A diagonal
    entry of R below tol * max is a rank-deficient aggregate (e.g. collinear nodes): an error naming it."""
    b = B.shape[1]
    free_nodes = np.flatnonzero(agg >= 0)
    order = np.argsort(agg[free_nodes], kind="stable")
    nodes_by_agg = free_nodes[order]
    starts = np.concatenate([[0], np.cumsum(np.bincount(agg[free_nodes], minlength=nagg))])
    wsum = np.bincount(agg[free_nodes], weights=weight[free_nodes], minlength=nagg)
    cen = np.stack([np.bincount(agg[free_nodes], weights=weight[free_nodes] * xyz[free_nodes, d], minlength=nagg)
                    for d in range(3)], axis=1) / wsum[:, None]
    S = np.tile(np.eye(6), (nagg, 1, 1))
    S[:, :3, 3:] = _rotations(cen - center)
    Sinv = S.copy()
    Sinv[:, :3, 3:] *= -1.0
    Q = np.zeros((agg.size, b, 6))
    R = np.zeros((nagg, 6, 6))
    for a in range(nagg):
        m = nodes_by_agg[starts[a]:starts[a + 1]]
        q, r = np.linalg.qr(B[m].reshape(-1, 6) @ Sinv[a])
        if q.shape[1] < 6:
            raise ValueError(f"AMG level {level}: aggregate {a} (nodes {m.tolist()}) has fewer than 6 dofs")
        s = np.where(np.diag(r) < 0, -1.0, 1.0)
        q, r = q * s[None, :], r * s[:, None]
        dg = np.abs(np.diag(r))
        if dg.min() < tol * dg.max():
            raise ValueError(f"AMG level {level}: aggregate {a} (nodes {m.tolist()}) has a rank-deficient rigid-body "
                             f"basis (R diagonal {dg.min():.3e} < {tol:g} x {dg.max():.3e})")
        Q[m] = q.reshape(m.size, b, 6)
        R[a] = r @ S[a]
    return Q[free_nodes], R, cen, wsum


def pair_lists(Aptr, Aind, Bptr, Bind, ncols):
    """Symbolic block product C = A B of two CSR block patterns.  Returns (Cptr, Cind, ptr, pa, pb): C's pattern, and
    for output block k the pairs (pa[t], pb[t]), t in [ptr[k], ptr[k+1]), ordered by A block then B block."""
    cnt = np.diff(Bptr)[Aind]
    tot = int(cnt.sum())
    pa = np.repeat(np.arange(Aind.size, dtype=np.int64), cnt)
    pb = np.repeat(Bptr[Aind], cnt) + (np.arange(tot, dtype=np.int64) - np.repeat(np.cumsum(cnt) - cnt, cnt))
    rowA = np.repeat(np.arange(Aptr.size - 1, dtype=np.int64), np.diff(Aptr))
    key = rowA[pa] * ncols + Bind[pb]
    del rowA
    order = np.argsort(key, kind="stable")
    key, pa, pb = key[order], pa[order].astype(np.int32), pb[order].astype(np.int32)
    del order
    first = np.flatnonzero(np.concatenate([[True], key[1:] != key[:-1]]))
    ukey = key[first]
    nrows = Aptr.size - 1
    Cptr = np.concatenate([[0], np.cumsum(np.bincount(ukey // ncols, minlength=nrows))]).astype(np.int64)
    return Cptr, ukey % ncols, np.append(first, tot).astype(np.int64), pa, pb


def transpose_pattern(ptr, ind, ncols):
    """(Tptr, Tind, idx): CSR pattern of the transpose and the gather map T block k = block idx[k] transposed."""
    nrows = ptr.size - 1
    rows = np.repeat(np.arange(nrows, dtype=np.int64), np.diff(ptr))
    idx = np.argsort(ind * nrows + rows, kind="stable")
    Tptr = np.concatenate([[0], np.cumsum(np.bincount(ind, minlength=ncols))]).astype(np.int64)
    return Tptr, rows[idx], idx


# --------------------------------------------------------------------------- device objects


def _t(a, dtype, dev):
    return torch.from_numpy(np.ascontiguousarray(a).astype(dtype)).to(dev)


class BSR:
    """Block-sparse matrix (br x bc blocks, row-major inside a block) on the device or the host."""

    def __init__(self, ptr, ind, br, bc, ncols, dev):
        self.br, self.bc, self.nbrows, self.nbcols = br, bc, ptr.size - 1, int(ncols)
        self.nnzb = int(ind.size)
        self.rowptr, self.colidx = _t(ptr, np.int32, dev), _t(ind, np.int32, dev)
        self.rowof = _t(np.repeat(np.arange(self.nbrows), np.diff(ptr)), np.int64, dev)
        self.vals = torch.zeros(self.nnzb * br * bc, dtype=torch.float64, device=dev)
        self._ptr_host, self._ind_host = ptr, ind

    @property
    def n(self):
        return self.nbrows * self.br

    def mult(self, x, y):
        if x.is_cuda:
            b2(lib.b200_bsr_spmv(self.br, self.bc, self.nbrows, self.rowptr.data_ptr(), self.colidx.data_ptr(),
                                 self.vals.data_ptr(), x.data_ptr(), y.data_ptr()))
            return
        prod = torch.bmm(self.vals.view(-1, self.br, self.bc), x.view(-1, self.bc)[self.colidx.long()].unsqueeze(2))
        y.zero_()
        y.view(-1, self.br).index_add_(0, self.rowof, prod.squeeze(2))

    def diag_positions(self):
        """value index of every diagonal entry, in row order (square block matrices with a diagonal block per row)"""
        rows = np.repeat(np.arange(self.nbrows), np.diff(self._ptr_host))
        blk = np.flatnonzero(rows == self._ind_host)
        assert blk.size == self.nbrows, "every block row needs its diagonal block"
        return (blk[:, None] * self.br * self.br + np.arange(self.br) * (self.br + 1)).reshape(-1)

    def to_scipy(self):
        """host copy as scipy.sparse.bsr_matrix (tests, reporting)"""
        import scipy.sparse as sp
        return sp.bsr_matrix((self.vals.cpu().numpy().reshape(-1, self.br, self.bc), self._ind_host, self._ptr_host),
                             shape=(self.nbrows * self.br, self.nbcols * self.bc))


class PairProduct:
    """C = A B over fixed pair lists (b200_bsr_pairs_product); optional smoothed-prolongator epilogue."""

    def __init__(self, ptr, pa, pb, br, bk, bc, dev):
        self.br, self.bk, self.bc, self.nout = br, bk, bc, ptr.size - 1
        self.ptr, self.pa, self.pb = _t(ptr, np.int64, dev), _t(pa, np.int32, dev), _t(pb, np.int32, dev)
        self.npairs = int(pa.size)

    def run(self, A, B, C, tmap=None, rowof=None, T=None, dinv=None, omega=None):
        if A.is_cuda:
            p = lambda t: t.data_ptr() if t is not None else None
            b2(lib.b200_bsr_pairs_product(self.br, self.bk, self.bc, self.nout, p(self.ptr), p(self.pa), p(self.pb),
                                          p(A), p(B), p(C), p(tmap), p(rowof), p(T), p(dinv), p(omega)))
            return
        prod = torch.bmm(A.view(-1, self.br, self.bk)[self.pa.long()], B.view(-1, self.bk, self.bc)[self.pb.long()])
        seg = torch.repeat_interleave(torch.arange(self.nout), torch.diff(self.ptr))
        out = torch.zeros((self.nout, self.br, self.bc), dtype=torch.float64)
        out.index_add_(0, seg, prod)
        if tmap is not None:
            t0 = torch.where((tmap >= 0)[:, None, None], T.view(-1, self.br, self.bc)[tmap.long().clamp_min(0)],
                             torch.zeros((), dtype=torch.float64))
            d = dinv.view(-1, self.br)[rowof.long()]
            out = t0 - omega[0] * d[:, :, None] * out
        C.copy_(out.reshape(-1))


def transpose_gather(src, dst, idx, br, bc):
    """dst blocks = src[idx] transposed (b200_bsr_transpose_gather)"""
    if src.is_cuda:
        b2(lib.b200_bsr_transpose_gather(br, bc, idx.numel(), idx.data_ptr(), src.data_ptr(), dst.data_ptr()))
    else:
        dst.copy_(src.view(-1, br, bc)[idx.long()].transpose(1, 2).reshape(-1))


class Level:
    """One level of the hierarchy: operator A (square BSR), and below the coarsest: the products to the next level."""


class SmoothedAggregationAMG:
    """Coarse solve of PMultigrid on the p = 1 level, on one device.

    dm: the LevelDM of the p = 1 level; mesh: its mesh (node_coords(1), offsets(1)).  The level-0 matrix lives on the
    L-vector layout (every node, 3 dofs); constrained (Dirichlet) rows and columns are masked with a unit diagonal and
    no aggregate contains a constrained node."""

    def __init__(self, dm, mesh, smooth_its=2, max_coarse=MAX_COARSE_DOFS, seed=200, elem_src=None):
        """elem_src: optional int array [mesh.nelem], element e -> its position in the element-matrix buffer the
        numeric set-up reads (default: position e).  RedundantAMG reads a rank-major gathered buffer this way."""
        t0 = time.perf_counter()
        if dm.halo is not None:
            raise NotImplementedError("SmoothedAggregationAMG takes the whole p = 1 level of one rank; partitioned runs "
                                      "use RedundantAMG")
        self.dm, dev = dm, dm.device
        self.device = dev
        en = mesh.offsets(1).reshape(-1, 8).astype(np.int64) // 3
        nn = dm.lsize // 3
        free = ~np.asarray(dm.bc_nodes, dtype=bool)
        gptr, gind = node_graph(en, nn)
        # level-0 pattern: the node graph without the couplings of constrained nodes; their rows keep the diagonal only
        rows = np.repeat(np.arange(nn), np.diff(gptr))
        keep = (rows == gind) | (free[rows] & free[gind])
        A0ptr = np.concatenate([[0], np.cumsum(np.bincount(rows[keep], minlength=nn))]).astype(np.int64)
        A0ind = gind[keep]
        del rows, keep
        # destination of every element-matrix block (e, row node a, column node b), both nodes free
        E = en.shape[0]
        a_, b_ = np.meshgrid(np.arange(8), np.arange(8), indexing="ij")
        rn, cn = en[:, a_.reshape(-1)], en[:, b_.reshape(-1)]                     # (E, 64)
        ok = free[rn] & free[cn]
        pos = np.arange(E, dtype=np.int64) if elem_src is None else np.asarray(elem_src, dtype=np.int64)
        src = ((pos[:, None] * 24 + 3 * b_.reshape(-1)[None, :]) * 24 + 3 * a_.reshape(-1)[None, :])
        keys0 = np.repeat(np.arange(nn, dtype=np.int64), np.diff(A0ptr)) * nn + A0ind
        dest = np.searchsorted(keys0, rn[ok] * nn + cn[ok])
        src = src[ok]
        del rn, cn, ok
        order = np.argsort(dest, kind="stable")
        self.e_ptr = _t(np.concatenate([[0], np.cumsum(np.bincount(dest, minlength=A0ind.size))]), np.int64, dev)
        self.e_src = _t(src[order], np.int64, dev)
        del dest, src, order
        cons = np.flatnonzero(~free)
        cons_blk = np.searchsorted(keys0, cons * nn + cons)
        self.ident_idx = _t((cons_blk[:, None] * 9 + np.array([0, 4, 8])).reshape(-1), np.int32, dev)
        self.ident_ones = torch.ones(self.ident_idx.numel(), dtype=torch.float64, device=dev)
        self._dense_idx = None
        del keys0

        coords = mesh.node_coords(1)
        self.center = coords[free].mean(axis=0) if free.any() else np.zeros(3)   # common centre of the rotations
        self.levels = []
        A = BSR(A0ptr, A0ind, 3, 3, nn, dev)
        node_free, b = free, 3
        stop = None
        self.near_null = [None]   # per coarse level: (nodes, 6, 6), column k = global rigid-body mode k at that node
        B, xyz, wgt = rigid_body_modes(coords, self.center), coords, np.ones(nn)
        agg_all = []
        while True:
            lev = Level()
            lev.A = A
            self.levels.append(lev)
            if A.n <= max_coarse:
                break
            if len(self.levels) >= MAX_LEVELS:
                stop = f"the level cap ({MAX_LEVELS})"
                break
            agg, nagg = aggregate(A._ptr_host, A._ind_host, node_free)
            if 6 * nagg * MIN_SHRINK > A.n:
                stop = f"aggregation shrinking it by less than {MIN_SHRINK:g}x ({A.n} -> {6 * nagg} rows)"
                break
            Qv, R, cen, w = tentative_prolongator(agg, nagg, B, xyz, wgt, self.center, level=len(self.levels) - 1)
            agg_all.append(agg)
            nrow = A.nbrows
            on = agg >= 0
            Tptr = np.concatenate([[0], np.cumsum(on.astype(np.int64))])
            Tind = agg[on]
            lev.Pt = BSR(Tptr, Tind, b, 6, nagg, dev)
            lev.Pt.vals.copy_(torch.from_numpy(Qv.reshape(-1)))
            # A P_tent -> P (same pattern); map P block -> P_tent block (or -1)
            Pptr, Pind, ptr1, pa1, pb1 = pair_lists(A._ptr_host, A._ind_host, Tptr, Tind, nagg)
            lev.P = BSR(Pptr, Pind, b, 6, nagg, dev)
            prow = np.repeat(np.arange(nrow), np.diff(Pptr))
            tmap = np.full(Pind.size, -1, dtype=np.int64)
            hit = on[prow] & (Pind == np.where(on, agg, -1)[prow])
            tmap[hit] = np.searchsorted(np.flatnonzero(on), prow[hit])
            lev.tmap = _t(tmap, np.int32, dev)
            lev.prow = _t(prow, np.int32, dev)
            lev.AP_t = PairProduct(ptr1, pa1, pb1, b, b, 6, dev)
            # P^T by a fixed gather
            PTptr, PTind, tidx = transpose_pattern(Pptr, Pind, nagg)
            lev.PT = BSR(PTptr, PTind, 6, b, nrow, dev)
            lev.tidx = _t(tidx, np.int32, dev)
            # A P, then A_c = P^T (A P)
            APptr, APind, ptr2, pa2, pb2 = pair_lists(A._ptr_host, A._ind_host, Pptr, Pind, nagg)
            lev.AP = BSR(APptr, APind, b, 6, nagg, dev)
            lev.AP_p = PairProduct(ptr2, pa2, pb2, b, b, 6, dev)
            Cptr, Cind, ptr3, pa3, pb3 = pair_lists(PTptr, PTind, APptr, APind, nagg)
            lev.Ac_p = PairProduct(ptr3, pa3, pb3, 6, b, 6, dev)
            del pa1, pb1, pa2, pb2, pa3, pb3
            A = BSR(Cptr, Cind, 6, 6, nagg, dev)
            node_free, b = np.ones(nagg, dtype=bool), 6
            B, xyz, wgt = R, cen, w
            self.near_null.append(R)
        self.aggregates = agg_all
        nc = self.levels[-1].A.n
        if nc > max_coarse:
            msg = (f"AMG: coarsening stopped at level {len(self.levels) - 1} with {nc} rows (target {max_coarse}) because "
                   f"of {stop}; the coarsest level is factored densely")
            if nc > MAX_DENSE_COARSEST:
                raise RuntimeError(f"{msg}, which at {nc} rows would need {16e-9 * nc * nc:.1f} GB (limit "
                                   f"{MAX_DENSE_COARSEST} rows)")
            warnings.warn(msg)
        L = len(self.levels)
        mk = lambda n: torch.zeros(n, dtype=torch.float64, device=dev)
        self.Vp = solver.Vec()          # private: AMG vector lengths must not pick up another level's dot weights
        for l, lev in enumerate(self.levels):
            n = lev.A.n
            lev.b, lev.x, lev.r, lev.t, lev.diag = mk(n), mk(n), mk(n), mk(n), mk(n)
            lev.diag_pos = _t(lev.A.diag_positions(), np.int32, dev)
            if l < L - 1:
                lev.sm = solver.ChebyshevJacobi(self.Vp, lev.A.mult, n, dev, smooth_its, seed=seed + l)
                lev.omega = mk(1)
        # coarsest level: dense inverse from a Cholesky factor, applied as a BSR with every block present
        C = self.levels[-1].A
        nb, bs = C.nbrows, C.br
        self.Cinv = BSR(np.arange(nb + 1, dtype=np.int64) * nb, np.tile(np.arange(nb), nb), bs, bs, nb, dev)
        rr = (C.rowof.cpu().numpy()[:, None, None] * bs + np.arange(bs)[None, :, None])
        cc = (C._ind_host[:, None, None] * bs + np.arange(bs)[None, None, :])
        self.dense_pos = _t((rr * C.n + cc).reshape(-1), np.int64, dev)
        self.cycles = 0
        self.symbolic_s = time.perf_counter() - t0

    # ---- numeric set-up (once per Newton step)
    def _assemble_level0(self, source):
        A0 = self.levels[0].A
        coo = getattr(source, "coo", None)
        if coo is not None:
            ev = coo.values()
            if ev.is_cuda:
                b2(lib.b200_bsr_assemble_elem(A0.nnzb, self.e_ptr.data_ptr(), self.e_src.data_ptr(), ev.data_ptr(),
                                              A0.vals.data_ptr()))
            else:
                off = torch.tensor([24 * j + i for i in range(3) for j in range(3)], dtype=torch.int64)
                g = ev[self.e_src[:, None] + off[None, :]]
                seg = torch.repeat_interleave(torch.arange(A0.nnzb), torch.diff(self.e_ptr))
                A0.vals.view(-1, 9).zero_().index_add_(0, seg, g)
        else:
            # CPU harness without element matrices: the operator probed column by column (SparseCoarseMatrix.dense)
            source.assemble()
            if getattr(source, "dense", None) is None:
                raise NotImplementedError("coarse='amg' needs the element matrices (assemble='coo') or a probed matrix")
            if self._dense_idx is None:
                n = self.dm.lsize
                rr = A0.rowof.cpu().numpy()[:, None, None] * 3 + np.arange(3)[None, :, None]
                cc = A0._ind_host[:, None, None] * 3 + np.arange(3)[None, None, :]
                self._dense_idx = _t((rr * n + cc).reshape(-1), np.int64, self.device)
            A0.vals.copy_(source.dense.reshape(-1)[self._dense_idx])
        if self.ident_idx.numel():
            if A0.vals.is_cuda:
                b2(lib.b200_scatter_set(A0.vals.data_ptr(), self.ident_idx.data_ptr(), self.ident_ones.data_ptr(),
                                        self.ident_idx.numel()))
            else:
                A0.vals[self.ident_idx.long()] = 1.0

    def _gather(self, dst, src, idx):
        if dst.is_cuda:
            b2(lib.b200_gather(dst.data_ptr(), src.data_ptr(), idx.data_ptr(), dst.numel()))
        else:
            dst.copy_(src[idx.long()])

    def setup(self, source):
        """source of the level-0 values: an object with .coo (CeedOperatorLinearAssemble element matrices, e.g. the
        p = 1 GpuLevel), or, without element matrices, a SparseCoarseMatrix that probes the operator (CPU harness)"""
        self._assemble_level0(source)
        for l, lev in enumerate(self.levels[:-1]):
            A = lev.A
            self._gather(lev.diag, A.vals, lev.diag_pos)
            lev.sm.setup(lev.diag)
            lev.omega.fill_(4.0 / (3.0 * (lev.sm.emax / 1.1)))        # omega = 4 / (3 lambda_max(D^-1 A))
            lev.AP_t.run(A.vals, lev.Pt.vals, lev.P.vals, tmap=lev.tmap, rowof=lev.prow, T=lev.Pt.vals,
                         dinv=lev.sm.dinv, omega=lev.omega)
            transpose_gather(lev.P.vals, lev.PT.vals, lev.tidx, lev.P.br, lev.P.bc)
            lev.AP_p.run(A.vals, lev.P.vals, lev.AP.vals)
            lev.Ac_p.run(lev.PT.vals, lev.AP.vals, self.levels[l + 1].A.vals)
        C = self.levels[-1].A
        dense = torch.zeros(C.n * C.n, dtype=torch.float64, device=self.device)
        dense[self.dense_pos] = C.vals
        dense = dense.view(C.n, C.n)
        inv = torch.cholesky_inverse(torch.linalg.cholesky(dense))
        nb, bs = C.nbrows, C.br
        self.Cinv.vals.copy_(inv.view(nb, bs, nb, bs).permute(0, 2, 1, 3).reshape(-1))

    # ---- the V-cycle
    def _cycle(self, l):
        V, lev = self.Vp, self.levels[l]
        if l == len(self.levels) - 1:
            self.Cinv.mult(lev.b, lev.x)
            return
        nxt = self.levels[l + 1]
        lev.sm.apply(lev.b, lev.x, zero_guess=True)
        lev.A.mult(lev.x, lev.t)
        V.axpby(lev.r, 1.0, lev.b, -1.0, lev.t)
        lev.PT.mult(lev.r, nxt.b)
        self._cycle(l + 1)
        lev.P.mult(nxt.x, lev.t)
        V.axpy(lev.x, 1.0, lev.t)
        lev.sm.apply(lev.b, lev.x, zero_guess=False)

    def solve(self, b, x):
        """x = one V-cycle applied to b (global vectors of the p = 1 level)"""
        self.dm.zero_and_global_to_local(b, self.levels[0].b)
        self._cycle(0)
        self.dm.local_to_global(self.levels[0].x, x)
        self.cycles += 1

    def level_info(self):
        """per level: rows and block nonzeros (and block shape)"""
        return [{"rows": lev.A.n, "nnzb": lev.A.nnzb, "block": lev.A.br} for lev in self.levels]

    def pair_counts(self):
        """pairs per product per level (A P_tent, A P, P^T A P)"""
        return [{"AP_tent": lev.AP_t.npairs, "AP": lev.AP_p.npairs, "PtAP": lev.Ac_p.npairs}
                for lev in self.levels[:-1]]


class RedundantAMG(SmoothedAggregationAMG):
    """The AMG coarse solve of a partitioned run (world > 1), as PETSc's PCREDUNDANT / GAMG process agglomeration:
    every rank builds and holds the whole hierarchy of the GLOBAL p = 1 level and applies it to the gathered
    right-hand side.

    dm, mesh: this rank's p = 1 LevelDM (masked layout) and part; gmesh: the global mesh, faces: the Dirichlet faces.
    Symbolic set-up (collective, once): the ranks' global element ids are exchanged and folded into the level-0
    assembly map, so b200_bsr_assemble_elem reads the gathered buffer directly.  Numeric set-up (once per Newton
    step): one all-gather of the element matrices into a rank-major buffer padded to the largest part.  Solve: the
    owned dofs of b are scattered into a zero global vector and summed over ranks (exact: one non-zero contribution
    per entry), one V-cycle runs on every rank, and each rank gathers its local dofs, shared ones included (the same
    bits on every holder).  Gathers are copies and the sum is exact, so every rank holds bit-identical levels."""

    def __init__(self, dm, mesh, gmesh, faces, dist, **kw):
        if not dm.masked:
            raise NotImplementedError("coarse='amg' with world > 1 needs the masked layout (masked=True)")
        self.dist, self.world = dist, dist.get_world_size()
        ids = [None] * self.world
        dist.all_gather_object(ids, np.asarray(mesh.elem_ids, dtype=np.int64))
        self.emax = max(v.size for v in ids)
        pos = np.full(gmesh.nelem, -1, dtype=np.int64)
        for r, v in enumerate(ids):
            if (pos[v] >= 0).any():
                raise ValueError(f"element(s) {v[pos[v] >= 0][:5].tolist()} are held by more than one rank")
            pos[v] = r * self.emax + np.arange(v.size)
        if (pos < 0).any():
            raise ValueError(f"{int((pos < 0).sum())} element(s) of the global mesh are held by no rank")
        from .matops import LevelDM
        dev = dm.device
        gdm = LevelDM(gmesh, 1, bc_faces=faces, device=dev, masked=True)
        super().__init__(gdm, gmesh, elem_src=pos, **kw)
        gnode = _global_node_ids(mesh, gmesh)
        gdof = (gnode[:, None] * 3 + np.arange(3)).reshape(-1)
        own = np.flatnonzero(np.repeat(dm.halo.owned_node_mask, 3))
        self.local_dm = dm
        self.l2g = _t(gdof, np.int32, dev)
        self.own_l, self.own_g = _t(own, np.int32, dev), _t(gdof[own], np.int32, dev)
        self.own_vals = torch.zeros(own.size, dtype=torch.float64, device=dev)
        self.bglob = torch.zeros(gdm.lsize, dtype=torch.float64, device=dev)
        self.xglob = torch.zeros(gdm.lsize, dtype=torch.float64, device=dev)
        self.send = torch.zeros(self.emax * 576, dtype=torch.float64, device=dev)
        self.gathered = torch.zeros(self.world * self.emax * 576, dtype=torch.float64, device=dev)
        self.coo = self            # setup() hands itself to SmoothedAggregationAMG.setup as the element-matrix source

    def values(self):
        return self.gathered

    def setup(self, source):
        """source: the p = 1 level with this rank's element matrices (.coo, CeedOperatorLinearAssemble layout)"""
        ev = source.coo.values()
        self.send[:ev.numel()].copy_(ev)
        if self.send.is_cuda:
            self.dist.all_gather_into_tensor(self.gathered, self.send)
        else:
            self.dist.all_gather(list(self.gathered.view(self.world, -1).unbind(0)), self.send)
        super().setup(self)

    def solve(self, b, x):
        """x = one V-cycle of the global hierarchy applied to b (masked local vectors of this rank's p = 1 level)"""
        self.bglob.zero_()
        self._gather(self.own_vals, b, self.own_l)
        if b.is_cuda:
            b2(lib.b200_scatter_set(self.bglob.data_ptr(), self.own_g.data_ptr(), self.own_vals.data_ptr(),
                                    self.own_vals.numel()))
        else:
            self.bglob[self.own_g.long()] = self.own_vals
        self.dist.all_reduce(self.bglob)
        super().solve(self.bglob, self.xglob)
        self._gather(x, self.xglob, self.l2g)


def _global_node_ids(mesh, gmesh):
    """global p = 1 node id of every local node of a part: HexSubMesh.node_ids, or a brick's lattice position"""
    if hasattr(mesh, "node_ids"):
        return mesh.node_ids(1)
    N, GN = mesh.nodes_per_dim(1), gmesh.nodes_per_dim(1)
    z, y, x = np.meshgrid(*(np.arange(N[d]) + mesh.origin[d] for d in (2, 1, 0)), indexing="ij")
    return (x + GN[0] * (y + GN[1] * z)).reshape(-1).astype(np.int64)
