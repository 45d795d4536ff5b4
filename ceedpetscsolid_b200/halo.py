"""Halo exchange for partitioned meshes: the PetscSF stand-in behind
DMGlobalToLocal(INSERT_VALUES) / DMLocalToGlobal(ADD_VALUES) (/root/reference/src/matops.c:33,57).

DMPlexDistribute with overlap 0 (/root/reference/src/setupdm.c:58-64) partitions ELEMENTS; mesh
nodes on partition interfaces are duplicated in the local vectors and owned by exactly one rank.
Here the partition is a grid of bricks of a box mesh (mesh.BoxMesh.brick) or a coordinate bisection of an
unstructured mesh (exodus.HexMesh.brick), and an interface node is owned by the LOWEST rank that holds it.
Two collective steps, both neighbour point-to-point (bricks: <= 26 neighbours, 7 for 2x2x2; at most 32):

  owner_to_ghost(Xloc)      owners send interface values, ghosts overwrite   (G2L, INSERT)
  ghost_to_owner_add(Yloc)  ghosts send partial sums, owners accumulate       (L2G, ADD)

Interface dofs are packed / unpacked with libceed_b200.so kernels (b200_gather,
b200_scatter_set, b200_scatter_add) and moved with torch.distributed batch_isend_irecv
(NCCL over NVLink for CUDA tensors, gloo for the CPU tests).
"""
import numpy as np
import torch


def _ranges(mesh_n, grid, p):
    """Per axis: node index range [lo, hi] (inclusive, global numbering) of every brick."""
    out = []
    for d in range(3):
        q, rem = divmod(mesh_n[d], grid[d])
        r = []
        for i in range(grid[d]):
            start = i * q + min(i, rem)
            size = q + (1 if i < rem else 0)
            r.append((start * p, (start + size) * p))
        out.append(r)
    return out


MAX_NEIGHBOURS = 32   # B200_HALO_MAX_NEIGHBOURS (include/b200_kernels.h)


def _brick_sets(gmesh, grid, rank, p):
    """Brick partition of a box: (local node count, shared {r: local node ids in global lexicographic order},
    owner [local node] = lowest rank holding it)."""
    px, py, pz = grid
    rng = _ranges(gmesh.n, grid, p)
    me = (rank % px, (rank // px) % py, rank // (px * py))
    lo = [rng[d][me[d]][0] for d in range(3)]
    hi = [rng[d][me[d]][1] for d in range(3)]
    N = [hi[d] - lo[d] + 1 for d in range(3)]  # local nodes per axis
    nnodes = N[0] * N[1] * N[2]
    owner = np.full((N[2], N[1], N[0]), rank, dtype=np.int64)
    shared = {}
    lidx = np.arange(nnodes).reshape(N[2], N[1], N[0])
    for dz in (-1, 0, 1):
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                if dx == dy == dz == 0:
                    continue
                nb = (me[0] + dx, me[1] + dy, me[2] + dz)
                if not all(0 <= nb[d] < grid[d] for d in range(3)):
                    continue
                r = nb[0] + px * (nb[1] + py * nb[2])
                sl = []
                for d, dd in enumerate((dx, dy, dz)):
                    # overlap of my node range with the neighbour's along axis d
                    a = max(lo[d], rng[d][nb[d]][0]); b = min(hi[d], rng[d][nb[d]][1])
                    assert a <= b
                    sl.append(slice(a - lo[d], b - lo[d] + 1))
                ids = lidx[sl[2], sl[1], sl[0]].reshape(-1)  # z,y,x order == global lexicographic order
                shared[r] = ids
                sub = owner[sl[2], sl[1], sl[0]]
                np.minimum(sub, r, out=sub)
    return nnodes, shared, owner.reshape(-1)


def _part_sets(gmesh, grid, rank, p):
    """Element partition of an unstructured mesh (exodus.HexMesh.brick): the same triple as _brick_sets, from the
    parts' global node ids at degree p.  A shared set lists its nodes in ascending global id, the same order on both
    sides; every rank computes this from the global mesh alone."""
    nodes = gmesh.part_node_ids(int(np.prod(grid)), p)
    mine = nodes[rank]
    owner = np.full(mine.size, rank, dtype=np.int64)
    shared = {}
    for r, other in enumerate(nodes):
        if r == rank:
            continue
        _, ids, _ = np.intersect1d(mine, other, assume_unique=True, return_indices=True)
        if ids.size:
            shared[r] = ids.astype(np.int64)
            np.minimum.at(owner, ids, r)
    return mine.size, shared, owner


class Halo:
    def __init__(self, gmesh, grid, rank, p, dist=None, device=None, ncomp=3):
        self.dist, self.rank, self.grid, self.p = dist, rank, grid, p
        sets = _brick_sets if getattr(gmesh, "structured", True) else _part_sets
        # shared[r] = local node indices (in a canonical GLOBAL order) shared with neighbour r
        self.nnodes, shared, own = sets(gmesh, grid, rank, p)
        self.neighbours = sorted(shared)
        if len(self.neighbours) > MAX_NEIGHBOURS:
            raise ValueError(f"rank {rank} shares nodes with {len(self.neighbours)} ranks; the halo exchange handles at "
                             f"most {MAX_NEIGHBOURS} neighbours")
        self.owned_node_mask = own == rank
        dev = device if device is not None else ("cuda" if torch.cuda.is_available() and dist is not None and dist.get_backend() == "nccl" else "cpu")
        self.device = torch.device(dev)

        def dofs(nodes):
            return (nodes[:, None] * ncomp + np.arange(ncomp)[None, :]).reshape(-1).astype(np.int32)

        # owner -> ghost: I send the nodes I own that r holds; I receive the nodes r owns
        # ghost -> owner: the reverse.  Both ranks enumerate a shared set in the same global order.
        self.send_own, self.recv_ghost = {}, {}
        for r in self.neighbours:
            ids = shared[r]
            mine = ids[own[ids] == rank]
            theirs = ids[own[ids] == r]
            if mine.size:
                self.send_own[r] = torch.from_numpy(dofs(mine)).to(self.device)
            if theirs.size:
                self.recv_ghost[r] = torch.from_numpy(dofs(theirs)).to(self.device)
        # one contiguous pack buffer per direction: a single gather kernel packs the data for ALL
        # neighbours, a single scatter kernel unpacks it; sends/receives are views into the buffers
        def layout(idx):
            ranks = [r for r in self.neighbours if r in idx]
            cat = torch.cat([idx[r] for r in ranks]) if ranks else torch.zeros(0, dtype=torch.int32, device=self.device)
            views, o = {}, 0
            for r in ranks:
                views[r] = (o, o + idx[r].numel())
                o += idx[r].numel()
            return cat.contiguous(), views

        self.own_cat, self.own_views = layout(self.send_own)
        self.ghost_cat, self.ghost_views = layout(self.recv_ghost)
        # "sum-and-share": every dof shared with r, both directions at once (same order on both sides)
        self.shared_all = {r: torch.from_numpy(dofs(shared[r])).to(self.device) for r in self.neighbours}
        self.share_cat, self.share_views = layout(self.shared_all)
        # canonical summation order of the sum-and-share: for every unique shared dof, the holders' partial sums in
        # ASCENDING RANK order, this rank's own (entry -1) included; the other entries are positions of the receive
        # buffer / window (laid out like share_cat).  Every holder then computes the bit-identical total.
        cat = self.share_cat.cpu().numpy().astype(np.int64)
        src_rank = np.concatenate([np.full(self.shared_all[r].numel(), r, dtype=np.int64) for r in self.neighbours]) \
            if self.neighbours else np.zeros(0, dtype=np.int64)
        udof = np.unique(cat)
        dof_all = np.concatenate([cat, udof])
        rank_all = np.concatenate([src_rank, np.full(udof.size, rank, dtype=np.int64)])
        ent_all = np.concatenate([np.arange(cat.size, dtype=np.int64), np.full(udof.size, -1, dtype=np.int64)])
        order = np.lexsort((rank_all, dof_all))
        counts = np.bincount(np.searchsorted(udof, dof_all), minlength=udof.size)
        uptr = np.zeros(udof.size + 1, dtype=np.int64)
        np.cumsum(counts, out=uptr[1:])
        self._udof_h, self._uptr_h, self._uent_h = udof, uptr, ent_all[order]
        self.udof = torch.from_numpy(udof.astype(np.int32)).to(self.device)
        self.uptr = torch.from_numpy(uptr.astype(np.int32)).to(self.device)
        self.uent = torch.from_numpy(self._uent_h.astype(np.int32)).to(self.device)
        self._ordered_cpu = None
        # number of ranks holding each local node (1 in the interior)
        cnt = np.ones(self.nnodes)
        for r in self.neighbours:
            cnt[shared[r]] += 1
        self.rank_multiplicity = cnt
        self._buf = {}

    def _buffer(self, key, n, like):
        k = (key, like.dtype, like.device)
        if k not in self._buf:
            self._buf[k] = torch.empty(n, dtype=like.dtype, device=like.device)
        return self._buf[k]

    @staticmethod
    def _gather(dst, src, idx):
        if idx.numel() == 0:
            return
        if src.is_cuda:
            from .ceed import b2, lib
            b2(lib.b200_gather(dst.data_ptr(), src.data_ptr(), idx.data_ptr(), idx.numel()))
        else:
            torch.index_select(src, 0, idx.long(), out=dst)

    @staticmethod
    def _scatter(dst, idx, src, add):
        if idx.numel() == 0:
            return
        if dst.is_cuda:
            from .ceed import b2, lib
            f = lib.b200_scatter_add if add else lib.b200_scatter_set
            b2(f(dst.data_ptr(), idx.data_ptr(), src.data_ptr(), idx.numel()))
        elif add:
            dst.index_add_(0, idx.long(), src)
        else:
            dst.index_copy_(0, idx.long(), src)

    def _exchange(self, vec, send_cat, send_views, recv_cat, recv_views, add, tag):
        dist = self.dist
        sbuf = self._buffer("s" + tag, send_cat.numel(), vec)
        rbuf = self._buffer("r" + tag, recv_cat.numel(), vec)
        self._gather(sbuf, vec, send_cat)
        ops = []
        for r in self.neighbours:  # same global order on every rank
            if r in recv_views:
                a, b = recv_views[r]
                ops.append(dist.P2POp(dist.irecv, rbuf[a:b], r))
            if r in send_views:
                a, b = send_views[r]
                ops.append(dist.P2POp(dist.isend, sbuf[a:b], r))
        if ops:
            for w in dist.batch_isend_irecv(ops):
                w.wait()
        if add is None:
            return rbuf
        self._scatter(vec, recv_cat, rbuf, add)

    def _unpack_ordered(self, Yloc, rbuf):
        """Yloc[shared dof] = sum of the holders' partial sums in ascending rank order (own partial sum = current value)."""
        if self.udof.numel() == 0:
            return
        if Yloc.is_cuda:
            from .ceed import b2, lib
            b2(lib.b200_halo_unpack_ordered(self.udof.numel(), self.udof.data_ptr(), self.uptr.data_ptr(),
                                            self.uent.data_ptr(), rbuf.data_ptr(), Yloc.data_ptr()))
            return
        if self._ordered_cpu is None:
            cnt = np.diff(self._uptr_h)
            pad = np.full((self._udof_h.size, int(cnt.max())), -2, dtype=np.int64)
            col = np.arange(self._uent_h.size) - np.repeat(self._uptr_h[:-1], cnt)
            pad[np.repeat(np.arange(self._udof_h.size), cnt), col] = self._uent_h
            self._ordered_cpu = (torch.from_numpy(self._udof_h), torch.from_numpy(pad))
        udof, pad = self._ordered_cpu
        own = Yloc[udof]
        s = torch.zeros_like(own)
        for k in range(pad.shape[1]):
            e = pad[:, k]
            s = s + torch.where(e == -1, own, torch.where(e >= 0, rbuf[e.clamp(min=0)], torch.zeros_like(own)))
        Yloc[udof] = s

    # ---- sum-and-share over NVLink peer memory (one node): no communication library on the data path
    def enable_p2p(self, timeout_s=None):
        """Collective over all ranks: allocate this rank's receive window, exchange CUDA IPC handles and segment
        layouts through torch.distributed (set-up only), map the neighbours' windows and create the C-side exchange
        object (csrc/b200_halo.cu).  Afterwards sum_and_share is push + signal on a high-priority side stream and
        wait + ordered unpack on the compute stream; `handle` can be given to CeedOperatorApplyPartitionedB200,
        which overlaps the exchange with the interior elements.  timeout_s (default $B200_HALO_TIMEOUT_S or 20):
        how long a rank waits for a neighbour before it flags the exchange as failed (check_p2p raises).
        Returns True when every rank succeeded; if any rank failed (no peer access, IPC refused ...) every rank
        releases what it set up and returns False, and the exchange keeps going through torch.distributed."""
        import os
        dist = self.dist
        assert self.device.type == "cuda", "peer-memory halo needs CUDA tensors"
        if timeout_s is None:
            timeout_s = float(os.environ.get("B200_HALO_TIMEOUT_S", "20"))
        import ctypes as C
        from .ceed import b2, lib

        def agree(err):
            """collective: did any rank fail this phase?"""
            flag = torch.tensor([0 if err is None else 1], dtype=torch.int32, device=self.device)
            dist.all_reduce(flag, op=dist.ReduceOp.MAX)
            if int(flag.item()):
                self._p2p_error = repr(err) if err is not None else "another rank could not set up its peer-memory window"
                self._release_p2p_local()
                return True
            return False

        # phase 1 (rank-local): allocate and export this rank's window
        total = int(self.share_cat.numel())
        err, handle = None, (C.c_ubyte * 64)()
        try:
            nbytes = int(lib.b200_halo_window_bytes(total))
            buf = C.c_void_p()
            b2(lib.b200_malloc(C.byref(buf), nbytes))
            self._p2p_buf = buf
            b2(lib.b200_memset(buf, 0, nbytes))
            b2(lib.b200_sync())
            b2(lib.b200_ipc_get_handle(buf, handle))
        except Exception as exc:
            err = exc
        if agree(err):
            return False
        # phase 2 (collective): everybody's handle and segment layout
        mine = {"rank": self.rank, "handle": bytes(handle), "total": total, "neighbours": list(self.neighbours),
                "views": {r: self.share_views[r] for r in self.neighbours}}
        infos = [None] * dist.get_world_size()
        dist.all_gather_object(infos, mine)
        # phase 3 (rank-local): map the neighbours' windows, create the exchange object
        try:
            self._map_neighbours(infos, total, timeout_s)
        except Exception as exc:
            err = exc
        if agree(err):
            return False
        dist.barrier()   # every window is mapped before anyone pushes
        return True

    def _release_p2p_local(self, barrier=None):
        """rank-local teardown (no collectives unless `barrier` is given: it is called between unmapping the
        neighbours' windows and freeing the own one, so that nobody frees memory a neighbour still has mapped)"""
        from .ceed import lib
        p = getattr(self, "_p2p", None)
        if p is not None and p.get("handle") is not None:
            lib.b200_halo_destroy(p["handle"])
        for base in getattr(self, "_p2p_open", []):
            lib.b200_ipc_close(base)
        self._p2p_open = []
        if barrier is not None:
            barrier()
        buf = getattr(self, "_p2p_buf", None)
        if buf is not None:
            lib.b200_sync()
            lib.b200_free(buf)
        self._p2p, self._p2p_buf = None, None

    def _map_neighbours(self, infos, total, timeout_s, bases=None):
        """bases: {neighbour rank: device address of its window} to use as they are, instead of opening the IPC
        handles of `infos` (windows that live in this process, e.g. several virtual ranks on one device)."""
        import ctypes as C
        from .ceed import b2, lib
        buf = self._p2p_buf
        nn = len(self.neighbours)
        seg_start = (C.c_int * (nn + 1))()
        remote = [(C.c_void_p * max(nn, 1))(), (C.c_void_p * max(nn, 1))()]   # per parity
        rflag = (C.c_void_p * max(nn, 1))()
        self._p2p_open = []
        for s, r in enumerate(self.neighbours):
            a, b = self.share_views[r]
            seg_start[s], seg_start[s + 1] = a, b
            info = infos[r]
            ra, rb = info["views"][self.rank]
            assert rb - ra == b - a, "shared sets of a rank pair must have the same size on both sides"
            if bases is None:
                opened = C.c_void_p()
                b2(lib.b200_ipc_open((C.c_ubyte * 64).from_buffer_copy(info["handle"]), C.byref(opened)))
                self._p2p_open.append(opened)
                base = opened.value
            else:
                base = int(bases[r])
            for par in (0, 1):
                remote[par][s] = base + (par * info["total"] + ra) * 8
            rflag[s] = base + 2 * info["total"] * 8 + info["neighbours"].index(self.rank) * 8
        h = C.c_void_p()
        b2(lib.b200_halo_create(nn, seg_start, remote[0], remote[1], rflag, self.share_cat.data_ptr(), total, buf,
                                self.udof.numel(), self.udof.data_ptr(), self.uptr.data_ptr(), self.uent.data_ptr(),
                                float(timeout_s), C.byref(h)))
        self._p2p = dict(buf=buf, handle=h)

    @property
    def handle(self):
        """b200_halo* of the peer-memory exchange (None unless enable_p2p was called)."""
        p = getattr(self, "_p2p", None)
        return p["handle"] if p is not None else None

    def check_p2p(self):
        """Raises if a peer-memory exchange ever timed out (synchronises the device)."""
        if getattr(self, "_p2p", None) is None:
            return
        import ctypes as C
        from .ceed import b2, lib
        e = C.c_int(0)
        b2(lib.b200_halo_error(self._p2p["handle"], C.byref(e)))
        if e.value:
            raise RuntimeError("peer-memory halo exchange timed out waiting for a neighbour: the vectors it produced "
                               "are incomplete")

    def p2p_failed_anywhere(self):
        """Collective: True if a peer-memory exchange timed out on ANY rank (synchronises)."""
        if getattr(self, "_p2p", None) is None:
            return False
        import ctypes as C
        from .ceed import b2, lib
        e = C.c_int(0)
        b2(lib.b200_halo_error(self._p2p["handle"], C.byref(e)))
        flag = torch.tensor([1 if e.value else 0], dtype=torch.int32, device=self.device)
        self.dist.all_reduce(flag, op=self.dist.ReduceOp.MAX)
        return bool(int(flag.item()))

    def close(self):
        """Collective: unmap the neighbours' windows and free this rank's (after every rank is done with them)."""
        if getattr(self, "_p2p", None) is None:
            return
        from .ceed import b2, lib
        b2(lib.b200_sync())
        self.dist.barrier()
        self._release_p2p_local(barrier=self.dist.barrier)

    def _sum_and_share_p2p(self, Yloc):
        from .ceed import b2, lib
        b2(lib.b200_halo_begin(self._p2p["handle"], Yloc.data_ptr()))
        b2(lib.b200_halo_end(self._p2p["handle"], Yloc.data_ptr()))

    def sum_and_share(self, Yloc):
        """One symmetric exchange replacing ghost->owner ADD followed by owner->ghost INSERT: every rank
        sends its partial sums on ALL shared dofs to every sharer and sums what it holds and receives in ascending
        rank order, so all copies end up with the same assembled value, bit for bit (SURVEY.md 8(e): allowed
        harness optimisation)."""
        if getattr(self, "_p2p", None) is not None and Yloc.is_cuda:
            return self._sum_and_share_p2p(Yloc)
        rbuf = self._exchange(Yloc, self.share_cat, self.share_views, self.share_cat, self.share_views, add=None, tag="sas")
        self._unpack_ordered(Yloc, rbuf)

    # ---- split form of sum_and_share: the exchange runs on a side stream while the caller keeps computing on
    # entries that are NOT shared (the interior elements of an operator application)
    def sum_and_share_begin(self, Yloc):
        """Pack the shared dofs (their partial sums must be complete) and start the neighbour exchange."""
        dist = self.dist
        sbuf = self._buffer("ssas", self.share_cat.numel(), Yloc)
        rbuf = self._buffer("rsas", self.share_cat.numel(), Yloc)
        self._gather(sbuf, Yloc, self.share_cat)
        ops = []
        for r in self.neighbours:
            a, b = self.share_views[r]
            ops.append(dist.P2POp(dist.irecv, rbuf[a:b], r))
            ops.append(dist.P2POp(dist.isend, sbuf[a:b], r))
        self._pending = None
        if not ops:
            return
        if Yloc.is_cuda:
            if getattr(self, "_side", None) is None:
                self._side = torch.cuda.Stream(device=Yloc.device)
                self._ev_packed = torch.cuda.Event()
                self._ev_recvd = torch.cuda.Event()
            self._ev_packed.record()                       # pack kernel queued on the compute stream
            self._side.wait_event(self._ev_packed)
            with torch.cuda.stream(self._side):
                works = dist.batch_isend_irecv(ops)
                for w in works:                            # stream-ordered wait: the host does not block
                    w.wait()
                self._ev_recvd.record()
            self._pending = ("cuda", rbuf)
        else:
            self._pending = ("cpu", rbuf, dist.batch_isend_irecv(ops))

    def sum_and_share_end(self, Yloc):
        """Wait for the exchange started by sum_and_share_begin and add the neighbours' partial sums."""
        pend, self._pending = self._pending, None
        if pend is None:
            return
        if pend[0] == "cuda":
            torch.cuda.current_stream(Yloc.device).wait_event(self._ev_recvd)
        else:
            for w in pend[2]:
                w.wait()
        self._unpack_ordered(Yloc, pend[1])

    def owner_to_ghost(self, Xloc):
        """DMGlobalToLocal part 2: ghosts receive the owner's value."""
        self._exchange(Xloc, self.own_cat, self.own_views, self.ghost_cat, self.ghost_views, add=False, tag="o2g")

    def ghost_to_owner_add(self, Yloc):
        """DMLocalToGlobal(ADD_VALUES) part 1: owners accumulate the ghosts' partial sums."""
        self._exchange(Yloc, self.ghost_cat, self.ghost_views, self.own_cat, self.own_views, add=True, tag="g2o")
