"""Loopback tests of the peer-memory halo exchange (csrc/b200_halo.cu) and of the overlapped partitioned operator apply
(CeedOperatorApplyPartitionedB200) with many virtual ranks on ONE GPU.

Every virtual rank's Halo is built by the production code.  Its receive window is an ordinary allocation on this
device, and Halo._map_neighbours(..., bases=...) maps the other virtual ranks' windows in place of the peer pointers
that CUDA IPC would give, so the real push, signal and wait-unpack kernels run with the production pointer and
flag-slot arithmetic.  The reference of an exchange is built from global node ids alone, not from the Halo tables:
for every global node held by several parts, s = 0.0 plus the holders' partial sums one by one in ascending rank
order, in float64.  Every holder must hold that value bit for bit; every other entry, and a few guard entries past
the end of each local vector, must be unchanged.

No wait kernel is ever queued before a push it needs: the GPU multiplexes streams onto a few hardware work queues, so
a spinning wait can hold back work queued after it on ANOTHER stream (issuing every virtual rank's partitioned apply
on its own stream and synchronising once timed out on 2 and 8 bricks).  Kernel-level tests therefore queue `begin`
for every rank and synchronise before any `end`.  Operator-level tests run the production partitioned apply on one
rank at a time, on its own stream, while the other ranks push their halo-free partial sums beforehand and finish the
exchange afterwards; every rank takes that role in turn.  The handles use a 5 s timeout and every test checks the
error word, so a scheduling problem fails the test instead of stalling it.

The tests without the gpu mark check the Halo sets and ordered-sum tables of a 34-part star against the global-id
reference, and the refusal of 33 neighbours.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from ceedpetscsolid_b200 import ceed
from ceedpetscsolid_b200.ceed import b2, lib
from ceedpetscsolid_b200.exodus import tube_mesh
from ceedpetscsolid_b200.halo import MAX_NEIGHBOURS, Halo
from ceedpetscsolid_b200.mesh import BoxMesh

ceed._proto("b200_get_stream", restype=ceed._vp)
ceed._proto("b200_halo_fork", ceed._vp, ceed._pvp)
ceed._proto("b200_halo_begin_forked", ceed._vp, ceed._vp)

GUARD = 5            # trailing entries of every local vector that no exchange may touch
TIMEOUT_S = 5.0
WRAP = 148 * 4 * 256  # entries past which the push and unpack grid-stride loops wrap


# ---------------------------------------------------------------------------------------------------- topologies
class StarMesh:
    """Duck-typed unstructured partition (what Halo needs of an exodus.HexMesh): part 0, the hub, shares a few
    thousand nodes with each of `nleaves` leaves; node "A" is held by the hub and every leaf, node "B" by all but the
    last leaf, so the last leaf shares exactly one node with every other leaf; neighbouring leaves share a few nodes,
    some also with the hub or with five holders; every part has private nodes, and one extra part holds nothing
    else (no neighbour).  Node ids are shuffled, so local and global order differ everywhere."""
    structured = False

    def __init__(self, nleaves=MAX_NEIGHBOURS, hub_share=1600, seed=0):
        self.nparts = nleaves + 2
        L = nleaves
        groups = [(1, range(L + 1)), (1, range(L))]
        groups += [(hub_share + (37 * l) % 101, (0, l)) for l in range(1, L + 1)]
        groups += [(1 + l % 3, (l, l + 1)) for l in range(1, L - 1)]
        groups += [(2, (0, l, l + 2)) for l in range(1, L - 2, 2)]
        groups += [(4, (0, 3, 7, 11, 19) if L > 19 else (0, 1, 2))]
        groups += [(3 + r % 5, (r,)) for r in range(self.nparts)]
        n = sum(c for c, _ in groups)
        M = np.zeros((n, self.nparts), dtype=bool)
        i = 0
        for c, holders in groups:
            M[i:i + c, list(holders)] = True
            i += c
        self.held = M[np.random.default_rng(seed).permutation(n)]   # held[global node, part]
        self.parts = [np.flatnonzero(self.held[:, r]) for r in range(self.nparts)]

    def part_node_ids(self, nparts, p):
        assert nparts == self.nparts
        return self.parts


def box_node_ids(gmesh, brick, p):
    """global lexicographic node id of every local node of a brick"""
    N, GN = brick.nodes_per_dim(p), gmesh.nodes_per_dim(p)
    ox, oy, oz = (brick.origin[d] * p for d in range(3))
    z, y, x = np.meshgrid(np.arange(N[2]) + oz, np.arange(N[1]) + oy, np.arange(N[0]) + ox, indexing="ij")
    return (x + GN[0] * (y + GN[1] * z)).reshape(-1)


def topology(name):
    """(global mesh, grid, degree, [global node ids of every rank's local nodes])"""
    if name == "star":
        m = StarMesh()
        return m, (m.nparts, 1, 1), 1, m.parts
    if name.startswith("tube"):
        m = tube_mesh(4, 32, 8, r0=0.6, r1=1.0, length=1.5)
        k = int(name[4:])
        return m, (k, 1, 1), 2, m.part_node_ids(k, 2)
    grid, n = {"box2": ((2, 1, 1), (6, 4, 4)), "box8": ((2, 2, 2), (6, 6, 6)), "box27": ((3, 3, 3), (9, 9, 9))}[name]
    m = BoxMesh(n=n, perturb=0.08, seed=0)
    return m, grid, 2, [box_node_ids(m, m.brick(grid, r), 2) for r in range(int(np.prod(grid)))]


def dofs(nodes):
    return (np.asarray(nodes, dtype=np.int64)[:, None] * 3 + np.arange(3)[None, :]).reshape(-1)


def holders_matrix(gids):
    """held[global node, rank]"""
    ng = 1 + max(int(g.max()) for g in gids if g.size)
    held = np.zeros((ng, len(gids)), dtype=bool)
    for r, g in enumerate(gids):
        held[g, r] = True
    return held


def ordered_sum_reference(gids, parts):
    """Expected vectors of a sum-and-share, from global ids: on every global dof held by several ranks, 0.0 plus the
    holders' partial sums in ascending rank order; every other entry (guards included) unchanged."""
    ng = 1 + max(int(g.max()) for g in gids if g.size)
    s, cnt = np.zeros(3 * ng), np.zeros(3 * ng, dtype=np.int64)
    for r, g in enumerate(gids):       # ascending rank
        d = dofs(g)
        s[d] = s[d] + parts[r][:d.size]
        cnt[d] += 1
    out = []
    for r, g in enumerate(gids):
        d = dofs(g)
        e = parts[r].copy()
        sh = cnt[d] > 1
        e[:d.size][sh] = s[d][sh]
        out.append(e)
    return out


def assert_bits(got, ref, what):
    got, ref = np.asarray(got), np.asarray(ref)
    bad = np.flatnonzero(got.view(np.int64) != ref.view(np.int64))
    assert bad.size == 0, f"{what}: {bad.size}/{ref.size} entries differ, first at {bad[:5]}: {got[bad[:5]]} != {ref[bad[:5]]}"


def check_tables(halo, gids, held):
    """The Halo's neighbour list, shared sets and ordered-sum tables of rank halo.rank against the global ids."""
    r = halo.rank
    g = gids[r]
    gd = dofs(g)
    sharers = np.flatnonzero(held[g].any(axis=0))
    assert halo.neighbours == [q for q in sharers.tolist() if q != r]
    cat = halo.share_cat.cpu().numpy().astype(np.int64)
    src = np.empty(cat.size, dtype=np.int64)
    for q in halo.neighbours:
        a, b = halo.share_views[q]
        src[a:b] = q
        assert np.array_equal(gd[cat[a:b]], dofs(np.intersect1d(g, gids[q]))), f"rank {r}: shared set with {q}"
    udof = halo.udof.cpu().numpy().astype(np.int64)
    uptr = halo.uptr.cpu().numpy().astype(np.int64)
    uent = halo.uent.cpu().numpy().astype(np.int64)
    multi = held[g].sum(axis=1) > 1
    assert np.array_equal(np.sort(gd[udof]), dofs(g[multi])), f"rank {r}: set of shared dofs"
    u_of = np.repeat(np.arange(udof.size), np.diff(uptr))
    exp_u, exp_rank = np.nonzero(held[gd[udof] // 3])     # row-major: holders of each shared dof in ascending rank
    assert np.array_equal(u_of, exp_u), f"rank {r}: holder counts"
    rank_of = np.where(uent < 0, r, src[np.maximum(uent, 0)])
    assert np.array_equal(rank_of, exp_rank), f"rank {r}: holders not in ascending rank order"
    gdof_of = np.where(uent < 0, gd[udof[u_of]], gd[cat[np.maximum(uent, 0)]])
    assert np.array_equal(gdof_of, gd[udof[u_of]]), f"rank {r}: a window entry of another dof"


# ---------------------------------------------------------------------------------------------------- CPU tests
def test_star_halo_tables_match_global_ids():
    m, grid, p, gids = topology("star")
    held = holders_matrix(gids)
    assert held.sum(axis=1).max() == MAX_NEIGHBOURS + 1
    halos = [Halo(m, grid, r, p, device="cpu") for r in range(m.nparts)]
    assert len(halos[0].neighbours) == MAX_NEIGHBOURS and halos[-1].neighbours == []
    assert all(len(h.neighbours) == MAX_NEIGHBOURS for h in halos[1:-1])
    last = halos[MAX_NEIGHBOURS]
    assert all(last.share_views[q][1] - last.share_views[q][0] == 3 for q in range(1, MAX_NEIGHBOURS))
    assert halos[0].share_cat.numel() > WRAP and halos[0].udof.numel() > WRAP
    for h in halos:
        check_tables(h, gids, held)


@pytest.mark.parametrize("name", ["box27", "tube12"])
def test_halo_tables_match_global_ids(name):
    m, grid, p, gids = topology(name)
    held = holders_matrix(gids)
    for r in range(len(gids)):
        check_tables(Halo(m, grid, r, p, device="cpu"), gids, held)
    if name == "box27":
        assert len(Halo(m, grid, 13, p, device="cpu").neighbours) == 26


def test_halo_refuses_33_neighbours():
    m = StarMesh(nleaves=MAX_NEIGHBOURS + 1, hub_share=2)
    with pytest.raises(ValueError, match="at most 32 neighbours"):
        Halo(m, (m.nparts, 1, 1), 0, 1, device="cpu")


def test_halo_create_refuses_33_neighbours():
    n = MAX_NEIGHBOURS + 1
    seg = (C.c_int * (n + 1))(*range(n + 1))
    ptrs = [(C.c_void_p * n)() for _ in range(3)]
    h = C.c_void_p()
    rc = lib.b200_halo_create(n, seg, ptrs[0], ptrs[1], ptrs[2], None, n, None, 0, None, None, None, 1.0, C.byref(h))
    assert rc != 0 and not h.value
    assert "too many neighbours" in lib.b200_last_error().decode()


# ---------------------------------------------------------------------------------------------------- loopback
class Loopback:
    """Every virtual rank's window allocated and zeroed on this device, and mapped into its neighbours' exchange
    objects by Halo._map_neighbours with the windows' own addresses as bases."""

    def __init__(self, halos, timeout_s=TIMEOUT_S):
        self.halos, self.stream0 = halos, lib.b200_get_stream()
        try:
            for h in halos:
                nbytes = int(lib.b200_halo_window_bytes(int(h.share_cat.numel())))
                buf = C.c_void_p()
                b2(lib.b200_malloc(C.byref(buf), C.c_size_t(nbytes)))
                h._p2p_buf = buf
                b2(lib.b200_memset(buf, 0, C.c_size_t(nbytes)))
            b2(lib.b200_sync())
            infos = [{"rank": h.rank, "total": int(h.share_cat.numel()), "neighbours": list(h.neighbours),
                      "views": {r: h.share_views[r] for r in h.neighbours}} for h in halos]
            for h in halos:
                h._map_neighbours(infos, infos[h.rank]["total"], timeout_s,
                                  bases={r: halos[r]._p2p_buf.value for r in h.neighbours})
        except BaseException:
            self.close()
            raise

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def check(self):
        """every handle's error word is 0 (synchronises)"""
        for h in self.halos:
            e = C.c_int(0)
            b2(lib.b200_halo_error(h.handle, C.byref(e)))
            assert e.value == 0, f"rank {h.rank}: a halo wait kernel timed out waiting for a neighbour's flag"

    def close(self):
        """synchronise, destroy every exchange object, then free every window; put the caller's stream back"""
        lib.b200_set_stream(self.stream0)
        torch.cuda.synchronize()
        for h in self.halos:
            p = getattr(h, "_p2p", None)
            if p is not None and p.get("handle") is not None:
                lib.b200_halo_destroy(p["handle"])
                p["handle"] = None
        for h in self.halos:
            h._release_p2p_local()


def loopback_topology(name):
    m, grid, p, gids = topology(name)
    halos = [Halo(m, grid, r, p, device="cuda") for r in range(len(gids))]
    return gids, halos


def fresh_parts(rng, gids):
    return [rng.standard_normal(3 * g.size + GUARD) for g in gids]


def to_device(parts):
    return [torch.from_numpy(v).cuda() for v in parts]


def exchange(halos, ys):
    for h, y in zip(halos, ys):
        b2(lib.b200_halo_begin(h.handle, y.data_ptr()))
    torch.cuda.synchronize()
    for h, y in zip(halos, ys):
        b2(lib.b200_halo_end(h.handle, y.data_ptr()))
    torch.cuda.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["box2", "box8", "box27", "tube6", "tube12", "star"])
def test_exchange_sums_holders_in_rank_order(name):
    gids, halos = loopback_topology(name)
    rng = np.random.default_rng(len(gids))
    with Loopback(halos) as lb:
        for it in range(5):   # both window parities, generations past 2
            parts = fresh_parts(rng, gids)
            ys = to_device(parts)
            exchange(halos, ys)
            for r, (y, ref) in enumerate(zip(ys, ordered_sum_reference(gids, parts))):
                assert_bits(y.cpu().numpy(), ref, f"{name} exchange {it}, rank {r}")
        lb.check()


@pytest.mark.gpu
def test_exchange_with_a_neighbour_one_exchange_ahead():
    """A pushes exchange g+1 into B's window (other parity, flag g+1) before B unpacks exchange g."""
    gids, halos = loopback_topology("box2")
    rng = np.random.default_rng(7)
    with Loopback(halos) as lb:
        for a, b in ((0, 1), (1, 0), (0, 1)):
            hA, hB = halos[a], halos[b]
            parts = fresh_parts(rng, gids)
            ys = to_device(parts)
            b2(lib.b200_halo_begin(hA.handle, ys[a].data_ptr()))
            b2(lib.b200_halo_begin(hB.handle, ys[b].data_ptr()))
            torch.cuda.synchronize()
            b2(lib.b200_halo_end(hA.handle, ys[a].data_ptr()))
            torch.cuda.synchronize()
            ref = ordered_sum_reference(gids, parts)
            assert_bits(ys[a].cpu().numpy(), ref[a], f"rank {a}, exchange g")
            nxt = fresh_parts(rng, gids)
            ys[a].copy_(torch.from_numpy(nxt[a]))
            b2(lib.b200_halo_begin(hA.handle, ys[a].data_ptr()))
            torch.cuda.synchronize()
            b2(lib.b200_halo_end(hB.handle, ys[b].data_ptr()))
            torch.cuda.synchronize()
            assert_bits(ys[b].cpu().numpy(), ref[b], f"rank {b}, exchange g after rank {a} pushed g+1")
            ys[b].copy_(torch.from_numpy(nxt[b]))
            b2(lib.b200_halo_begin(hB.handle, ys[b].data_ptr()))
            torch.cuda.synchronize()
            b2(lib.b200_halo_end(hA.handle, ys[a].data_ptr()))
            b2(lib.b200_halo_end(hB.handle, ys[b].data_ptr()))
            torch.cuda.synchronize()
            for r, ref in enumerate(ordered_sum_reference(gids, nxt)):
                assert_bits(ys[r].cpu().numpy(), ref, f"rank {r}, exchange g+1")
        lb.check()


@pytest.mark.gpu
@pytest.mark.parametrize("name,rank", [("box27", 13), ("star", 0), ("star", MAX_NEIGHBOURS + 1)])
def test_forked_exchange_sees_the_side_stream_writes(name, rank):
    """b200_halo_fork; the partial sums of `rank` are produced on the side stream (a long b200_vec_scale); then
    begin_forked and end on the compute stream, and a copy queued right after end must see the scaled values.
    The other ranks push first and are synchronised, so the wait kernel of `rank` never waits for later work."""
    gids, halos = loopback_topology(name)
    tail = 1 << 26             # ~0.5 GB scaled behind the partial sums: the side-stream kernel takes visible time
    rng = np.random.default_rng(rank + 3)
    h = halos[rank]
    others = [q for q in range(len(halos)) if q != rank]
    with Loopback(halos) as lb:
        for it in range(3):
            parts = fresh_parts(rng, gids)
            ys = to_device(parts)
            big = torch.empty(parts[rank].size + tail, dtype=torch.float64, device="cuda")
            big[:parts[rank].size] = ys[rank]
            big[parts[rank].size:] = 1.0
            ys[rank] = big
            for q in others:
                b2(lib.b200_halo_begin(halos[q].handle, ys[q].data_ptr()))
            torch.cuda.synchronize()
            side = C.c_void_p()
            b2(lib.b200_halo_fork(h.handle, C.byref(side)))
            b2(lib.b200_set_stream(side))
            b2(lib.b200_vec_scale(big.data_ptr(), 0.5, big.numel()))
            b2(lib.b200_set_stream(lb.stream0))
            b2(lib.b200_halo_begin_forked(h.handle, big.data_ptr()))
            b2(lib.b200_halo_end(h.handle, big.data_ptr()))
            seen = big.clone()        # compute stream, right behind end
            torch.cuda.synchronize()
            for q in others:
                b2(lib.b200_halo_end(halos[q].handle, ys[q].data_ptr()))
            torch.cuda.synchronize()
            parts[rank] = parts[rank] * 0.5
            ref = ordered_sum_reference(gids, parts)
            assert_bits(seen[:parts[rank].size].cpu().numpy(), ref[rank], f"{name} rank {rank} (forked), {it}")
            assert bool((seen[parts[rank].size:] == 0.5).all()), "the copy behind end ran before the side stream's work"
            for q in others:
                assert_bits(ys[q].cpu().numpy(), ref[q], f"{name} rank {q}, {it}")
        lb.check()


# ---------------------------------------------------------------------------------------------------- operators
OP_TOPOS = {"box2": ((2, 1, 1), (8, 4, 4)), "box8": ((2, 2, 2), (8, 8, 8)), "box27": ((3, 3, 3), (18, 18, 18)),
            "tube6": ((6, 1, 1), None)}
_oracles = {}


def op_global(name):
    grid, n = OP_TOPOS[name]
    m = tube_mesh(4, 32, 8, r0=0.6, r1=1.0, length=1.5) if n is None else BoxMesh(n=n, perturb=0.08, seed=0)
    return m, grid, n


def oracle_for(name, problem, p):
    """(OracleProblem of the global mesh, global Dirichlet dof mask), cached per case"""
    key = (name, problem, p)
    if key not in _oracles:
        from helpers import OracleProblem
        m, _, n = op_global(name)
        o = OracleProblem(problem, n, p) if n is not None else OracleProblem(problem, None, p, mesh=m)
        _oracles[key] = (o, np.repeat(o.mesh.boundary_mask(p, "all"), 3))
    return _oracles[key]


class OpRank:
    """One virtual rank: its own Ceed (the deterministic E-vector scratch belongs to the Ceed), the fine level of
    setup_all on its interface-first brick, the masked LevelDM, its own non-blocking stream."""

    def __init__(self, gmesh, grid, r, problem, p, resource):
        from ceedpetscsolid_b200 import matops, setuplibceed
        from ceedpetscsolid_b200.mesh import smooth_displacement
        self.rank = r
        self.mesh = mesh = gmesh.brick(grid, r, interface_first=True)
        self.ceed = ceed.Ceed(resource)
        _, data, _ = setuplibceed.setup_all(self.ceed, mesh, problem, p, multigrid="none")
        self.data = data[-1]
        self.halo = Halo(gmesh, grid, r, p, device="cuda")
        self.dm = matops.LevelDM(mesh, p, bc_faces="all", halo=self.halo, masked=True)
        gids = box_node_ids(gmesh, mesh, p) if getattr(gmesh, "structured", True) else mesh.node_ids(p)
        self.gdof = dofs(gids)
        self.stream = torch.cuda.Stream()
        n = mesh.lsize(p)
        self.xc, self.yc = self.ceed.Vector(n), self.ceed.Vector(n)
        self.u = torch.from_numpy(smooth_displacement(mesh.node_coords(p)).reshape(-1)).cuda()
        self.X, self.Y = torch.zeros_like(self.u), torch.zeros_like(self.u)
        # first-launch set-up (gradu, Jacobian cache, scratch) before any loopback handle exists
        self.apply(self.data.opApply, self.u, self.Y, 0, None, None)
        self.apply(self.data.opJacob, self.u, self.Y, 0, None, None)
        torch.cuda.synchronize()

    def apply(self, op, x, y, nif, handle, mask):
        self.xc.set_array(x)
        self.yc.set_array(y)
        op.apply_partitioned(self.xc, self.yc, nif, handle, mask)
        self.xc.take_array()
        self.yc.take_array()

    def gradu(self):
        return self.data.gradu.to_numpy()


def op_ranks(name, problem, p, resource):
    gmesh, grid, _ = op_global(name)
    return gmesh, [OpRank(gmesh, grid, r, problem, p, resource) for r in range(int(np.prod(grid)))]


def run_subject(ranks, subject, op_of, x_of, nif):
    """One exchange in which rank `subject` runs the production CeedOperatorApplyPartitionedB200 on its own stream and
    every other rank runs its halo-free local apply, pushes it (b200_halo_begin) and is synchronised first; those ranks
    then finish the exchange (b200_halo_end) and zero their Dirichlet rows.  So the subject's wait kernel finds every
    flag raised, and no wait kernel is ever queued before a push it needs: streams share the GPU's hardware work
    queues, and a spinning wait can hold back work queued after it on another stream.  Returns the local partial sums
    of the other ranks (None for the subject)."""
    local = []
    for rk in ranks:
        if rk.rank != subject:
            rk.apply(op_of(rk), x_of(rk), rk.Y, 0, None, None)
    torch.cuda.synchronize()
    for rk in ranks:
        local.append(None if rk.rank == subject else rk.Y.cpu().numpy())
        if rk.rank != subject:
            b2(lib.b200_halo_begin(rk.halo.handle, rk.Y.data_ptr()))
    torch.cuda.synchronize()
    rk = ranks[subject]
    s0 = lib.b200_get_stream()
    try:
        rk.ceed.set_stream(rk.stream.cuda_stream)
        rk.apply(op_of(rk), x_of(rk), rk.Y, nif, rk.halo.handle, rk.dm.bc_idx)
    finally:
        lib.b200_set_stream(s0)
    torch.cuda.synchronize()
    for rk in ranks:
        if rk.rank != subject:
            b2(lib.b200_halo_end(rk.halo.handle, rk.Y.data_ptr()))
            rk.dm.zero_constrained(rk.Y)
    torch.cuda.synchronize()
    return local


def check_against_oracle(ranks, outs, yref, gbc, what):
    """to 1e-12 relative on free dofs, Dirichlet rows exactly 0, every interface copy bit-identical"""
    from helpers import rel_err
    ypar = np.full(yref.size, np.nan)
    seen = np.zeros(yref.size, dtype=np.int64)
    for rk, v in zip(ranks, outs):
        d = rk.gdof
        again = seen[d] > 0
        assert_bits(v[again], ypar[d][again], f"{what}: interface copies of rank {rk.rank}")
        assert np.all(v[gbc[d]] == 0.0), f"{what}: a Dirichlet row of rank {rk.rank} is not 0"
        ypar[d] = v
        seen[d] += 1
    free = ~gbc
    assert np.all(seen >= 1)
    err = rel_err(ypar[free], yref[free])
    assert err < 1e-12, f"{what}: relative error {err:.3e} against the oracle"


def subjects(ranks):
    """the rank with the most neighbours first, then every other rank"""
    hub = max(range(len(ranks)), key=lambda r: (len(ranks[r].halo.neighbours), -r))
    return [hub] + [r for r in range(len(ranks)) if r != hub]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["default", "deterministic"])
@pytest.mark.parametrize("name", ["box2", "box8", "box27", "tube6"])
@pytest.mark.parametrize("problem,p", [("hyperFS", 2), ("hyperFS", 4), ("hyperSS", 3)])
def test_partitioned_jacobian_loopback(problem, p, name, mode):
    """Jacobian MatMult through CeedOperatorApplyPartitionedB200 on every virtual rank in turn, overlapped
    (0 < n_interface < nelem) and not (n_interface = 0), against the serial oracle; in deterministic mode also
    bitwise against the rank's own halo-free apply + the ordered sum by global id, with the masked rows zeroed."""
    o, gbc = oracle_for(name, problem, p)
    gmesh, ranks = op_ranks(name, problem, p, "/gpu/b200" + (":deterministic" if mode == "deterministic" else ""))
    assert all(0 < rk.mesh.n_interface < rk.mesh.nelem for rk in ranks)
    gids = [rk.gdof[::3] // 3 for rk in ranks]
    rng = np.random.default_rng(p)
    order = subjects(ranks)
    with Loopback([rk.halo for rk in ranks]) as lb:
        for overlap in (True, False):
            for it in range(3):
                xg = rng.standard_normal(gbc.size)
                xg[gbc] = 0.0
                yref = o.jacobian(xg)
                for rk in ranks:
                    rk.X.copy_(torch.from_numpy(xg[rk.gdof]))
                torch.cuda.synchronize()
                for subject in (order if it == 0 else order[:1] + order[1 + it::3]):
                    rk = ranks[subject]
                    nif = rk.mesh.n_interface if overlap else 0
                    local = run_subject(ranks, subject, lambda rk: rk.data.opJacob, lambda rk: rk.X, nif)
                    lb.check()
                    outs = [rk.Y.cpu().numpy() for rk in ranks]
                    what = (f"{problem} p={p} {name} {mode}, rank {subject} with n_interface={nif} of "
                            f"{rk.mesh.nelem}, x {it}")
                    check_against_oracle(ranks, outs, yref, gbc, what)
                    if mode == "deterministic":
                        z = torch.zeros_like(rk.Y)
                        rk.apply(rk.data.opJacob, rk.X, z, 0, None, None)
                        local[subject] = z.cpu().numpy()
                        ref = ordered_sum_reference(gids, local)[subject]
                        ref[rk.dm.bc_idx.cpu().numpy()] = 0.0
                        assert_bits(outs[subject], ref, f"{what}: against its own apply + the ordered sum")


@pytest.mark.gpu
def test_partitioned_fused_residual_loopback():
    """The fused residual through CeedOperatorApplyPartitionedB200 with an overlapped split (interface elements on the
    side stream, interior on the compute stream, both writing their slices of gradu), every rank in turn: the output
    against the oracle residual, gradu (NaN beforehand) bitwise equal to a plain CeedOperatorApply on the same rank,
    and a following partitioned Jacobian against the oracle."""
    name, problem, p = "box8", "hyperFS", 2
    o, gbc = oracle_for(name, problem, p)
    gmesh, ranks = op_ranks(name, problem, p, "/gpu/b200")
    rres = o.residual_fine(o.u_fine)
    xg = np.random.default_rng(1).standard_normal(gbc.size)
    xg[gbc] = 0.0
    yjac = o.jacobian(xg)
    for rk in ranks:
        rk.X.copy_(torch.from_numpy(xg[rk.gdof]))
    with Loopback([rk.halo for rk in ranks]) as lb:
        for subject in subjects(ranks):
            rk = ranks[subject]
            rk.data.gradu.set_value(float("nan"))
            torch.cuda.synchronize()
            run_subject(ranks, subject, lambda rk: rk.data.opApply, lambda rk: rk.u, rk.mesh.n_interface)
            lb.check()
            check_against_oracle(ranks, [q.Y.cpu().numpy() for q in ranks], rres, gbc,
                                 f"partitioned residual on rank {subject}")
            g = rk.gradu()
            assert not np.isnan(g).any(), f"rank {subject}: an element range left its slice of gradu unwritten"
            run_subject(ranks, subject, lambda rk: rk.data.opJacob, lambda rk: rk.X, rk.mesh.n_interface)
            lb.check()
            check_against_oracle(ranks, [q.Y.cpu().numpy() for q in ranks], yjac, gbc,
                                 f"Jacobian after the partitioned residual on rank {subject}")
            r = torch.zeros_like(rk.Y)
            rk.xc.set_array(rk.u)
            rk.yc.set_array(r)
            rk.data.opApply.apply(rk.xc, rk.yc)
            rk.xc.take_array()
            rk.yc.take_array()
            assert_bits(g, rk.gradu(), f"rank {subject}: gradu of the partitioned residual vs a plain apply")
