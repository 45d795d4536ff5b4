"""Unstructured hex meshes on several ranks (CPU, gloo): the coordinate-bisection partition (exodus.HexMesh.brick), the
halo sets built from the parts' global node ids, Dirichlet masks restricted from the global mesh, the partitioned
oracle apply, the partitioned Newton-Krylov-p-MG solve, and the redundant AMG coarse solve (amg.RedundantAMG)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from ceedpetscsolid_b200.exodus import tube_mesh
from ceedpetscsolid_b200.halo import Halo
from ceedpetscsolid_b200.mesh import grid_for


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _mesh(kind):
    """closed tube: the angular seam shares vertices; open sector: no seam"""
    if kind == "tube":
        return tube_mesh(2, 16, 6, r0=0.6, r1=1.0, length=1.5)
    return tube_mesh(2, 12, 6, r0=0.6, r1=1.0, length=1.5, angle=np.pi)


def _spawn(fn, world, *args):
    mp.spawn(fn, args=(world, _free_port()) + args, nprocs=world, join=True)


def _init(rank, world, port):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)


def _dofs(nodes, ncomp=3):
    return (np.asarray(nodes)[:, None] * ncomp + np.arange(ncomp)[None, :]).reshape(-1)


# --------------------------------------------------------------------------- partition, halo sets, masks (no ranks)


@pytest.mark.parametrize("kind", ["tube", "sector"])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_partition_covers_every_element_once_is_reproducible_and_puts_the_interface_first(kind, world):
    m = _mesh(kind)
    parts = m.partition(world)
    allel = np.concatenate(parts)
    assert len(parts) == world and min(p.size for p in parts) > 0
    assert np.array_equal(np.sort(allel), np.arange(m.nelem))
    assert max(p.size for p in parts) - min(p.size for p in parts) <= 1            # counts in proportion
    again = _mesh(kind).partition(world)                                             # fresh mesh object, no cache
    assert all(np.array_equal(a, b) for a, b in zip(parts, again))
    held = np.zeros(m.vertices.shape[0], dtype=int)
    for p in parts:
        held[np.unique(m.connect[p])] += 1
    for r in range(world):
        plain, first = m.brick(grid_for(world), r), m.brick(grid_for(world), r, interface_first=True)
        assert np.array_equal(plain.elem_ids, parts[r]) and plain.elem_order is None
        assert np.array_equal(first.elem_ids, plain.elem_ids[first.elem_order])
        for p in (1, 2, 3):
            assert np.array_equal(first.offsets(p), plain.offsets(p)[first.elem_order])
            assert np.array_equal(first.node_ids(p), plain.node_ids(p))
        touch = (held[m.connect[first.elem_ids]] > 1).any(axis=1)
        nif = first.n_interface
        assert touch.any() and not touch[nif:].any() and touch[:int(touch.sum())].all()
        assert nif % 16 == 0 or nif == first.nelem
        # the part's local mesh is the parent's restricted: same vertices, same nodes at every degree
        assert np.array_equal(plain.coord_lvector().reshape(-1, 3), m.vertices[plain.node_ids(1)])
        for p in (1, 2):
            gids = m._level(p)[0][plain.elem_ids]
            assert np.array_equal(plain.node_ids(p)[plain.offsets(p) // 3], gids)


@pytest.mark.parametrize("kind", ["tube", "sector"])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_halo_sets_are_symmetric_owned_by_the_lowest_holder_and_count_the_holders(kind, world):
    m = _mesh(kind)
    grid = grid_for(world)
    for p in (1, 2):
        subs = [m.brick(grid, r) for r in range(world)]
        halos = [Halo(m, grid, r, p, device="cpu") for r in range(world)]
        holders = {}
        for r, s in enumerate(subs):
            for g in s.node_ids(p):
                holders.setdefault(int(g), []).append(r)
        for r, (s, h) in enumerate(zip(subs, halos)):
            gid = s.node_ids(p)
            assert h.nnodes == gid.size
            nb = sorted({q for g in gid for q in holders[int(g)] if q != r})
            assert h.neighbours == nb
            for q in nb:
                mine = gid[h.shared_all[q].numpy()[::3] // 3]
                theirs = subs[q].node_ids(p)[halos[q].shared_all[r].numpy()[::3] // 3]
                assert np.array_equal(mine, theirs) and np.all(np.diff(mine) > 0)     # same ids, same order
            owner = np.array([min(holders[int(g)]) for g in gid])
            assert np.array_equal(h.owned_node_mask, owner == r)
            assert np.array_equal(h.rank_multiplicity, [len(holders[int(g)]) for g in gid])
        if kind == "tube":   # the seam: nodes at angle 0 are shared by the parts on both sides of it
            assert any(len(v) > 1 for v in holders.values())


def test_dirichlet_node_held_only_through_an_edge_is_masked_on_every_holder():
    """side set 3 = the z = 0 faces of part 0's elements only: part 1 holds nodes of it through element edges and owns
    none of its faces, and still masks them"""
    m = tube_mesh(2, 16, 4)
    parts = m.partition(2)
    el = np.intersect1d(parts[0], m.sidesets[1][0])
    m.sidesets[3] = (el, np.full(el.size, 5))
    assert np.intersect1d(m.sidesets[3][0], parts[1]).size == 0
    for p in (1, 2, 3):
        gmask = m.boundary_mask(p, [3])
        for r in range(2):
            s = m.brick((2, 1, 1), r)
            assert np.array_equal(s.boundary_mask(p, [3]), gmask[s.node_ids(p)])
        s1 = m.brick((2, 1, 1), 1)
        assert s1.boundary_mask(p, [3]).any()


def test_more_neighbours_than_the_halo_handles_is_an_error(monkeypatch):
    import ceedpetscsolid_b200.halo as halo_mod
    monkeypatch.setattr(halo_mod, "MAX_NEIGHBOURS", 1)
    m = _mesh("tube")
    with pytest.raises(ValueError, match="at most 1 neighbours"):
        Halo(m, grid_for(8), 0, 1, device="cpu")


# --------------------------------------------------------------------------- partitioned oracle apply (gloo)


def _apply_worker(rank, world, port, kind, p, out):
    _init(rank, world, port)
    try:
        from helpers import PHYS
        from oracle import oracle
        m = _mesh(kind)
        grid = grid_for(world)
        sub = m.brick(grid, rank, interface_first=True)
        halo = Halo(m, grid, rank, p, dist, device="cpu")
        gdof = _dofs(sub.node_ids(p))
        P = Q = p + 1
        B, D, _, _ = oracle.basis_1d(P, Q, 0)
        qdata = oracle.setup_geo(sub.nelem, Q, sub.offsets(1), sub.coord_lvector())
        xg = np.random.default_rng(3).standard_normal(m.lsize(p))
        # shared layout: every copy of x, one sum-and-share
        y = torch.from_numpy(oracle.operator_apply("linElas", True, PHYS, sub.nelem, P, Q, B, D, sub.offsets(p), qdata,
                                                   None, xg[gdof].copy()))
        y_owner = y.clone()
        halo.sum_and_share(y)
        # owner/ghost layout: ghosts add into the owner, the owner sends the total back
        halo.ghost_to_owner_add(y_owner)
        halo.owner_to_ghost(y_owner)
        np.savez(os.path.join(out, f"a{rank}.npz"), gdof=gdof, y=y.numpy(), y_owner=y_owner.numpy(),
                 mult=np.repeat(halo.rank_multiplicity, 3))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,kind,p", [(2, "tube", 1), (4, "tube", 2), (8, "tube", 3),
                                          (2, "sector", 3), (4, "sector", 1), (8, "sector", 2)])
def test_partitioned_oracle_apply_matches_serial(tmp_path, world, kind, p):
    from helpers import PHYS
    from oracle import oracle
    _spawn(_apply_worker, world, kind, p, str(tmp_path))
    m = _mesh(kind)
    P = Q = p + 1
    B, D, _, _ = oracle.basis_1d(P, Q, 0)
    qdata = oracle.setup_geo(m.nelem, Q, m.offsets(1), m.coord_lvector())
    xg = np.random.default_rng(3).standard_normal(m.lsize(p))
    yser = oracle.operator_apply("linElas", True, PHYS, m.nelem, P, Q, B, D, m.offsets(p), qdata, None, xg)
    first = np.full(yser.size, np.nan)
    holders = np.zeros(yser.size)
    for r in range(world):
        d = np.load(tmp_path / f"a{r}.npz")
        gd = d["gdof"]
        assert np.linalg.norm(d["y"] - yser[gd]) <= 1e-13 * np.linalg.norm(yser)
        assert np.linalg.norm(d["y_owner"] - yser[gd]) <= 1e-13 * np.linalg.norm(yser)
        seen = ~np.isnan(first[gd])
        assert np.array_equal(d["y"][seen], first[gd][seen]), f"rank {r}: interface copies differ bitwise"
        first[gd] = d["y"]
        np.add.at(holders, gd, 1.0 / d["mult"])
    np.testing.assert_allclose(holders, 1.0, atol=1e-14)


# --------------------------------------------------------------------------- partitioned solves (gloo)


def _app():
    from ceedpetscsolid_b200.elasticity import AppCtx
    m = tube_mesh(2, 12, 6, r0=0.6, r1=1.0, length=1.5)
    return AppCtx(problem="hyperFS", degree=2, num_steps=1, mesh=m,
                  clamp={1: [0, 0, 0, 0, 0, 1, 0], 2: [0.02, 0, -0.05, 0, 0, 1, 0.05]})


def _amg_oracle_solve(app, dist_, rank, world):
    """oracle_levels.oracle_solve with an AMG coarse solve from the (fixed) oracle element matrices of the p = 1 level:
    SmoothedAggregationAMG on one rank, RedundantAMG on several"""
    from ceedpetscsolid_b200 import matops, solver
    from ceedpetscsolid_b200.amg import RedundantAMG, SmoothedAggregationAMG
    from amg_helpers import Coo, oracle_element_matrices
    from oracle_levels import OracleLevel, OracleShared, OracleTransfer
    sh = OracleShared(app, True, dist_, rank, world)
    L = len(sh.degrees)
    levels = [OracleLevel(sh, l, l == L - 1) for l in range(L)]
    transfers = [None] + [OracleTransfer(sh, levels[l - 1], levels[l]) for l in range(1, L)]
    levels[0].coo = Coo(sh.mesh, oracle_element_matrices(sh.mesh))
    V = solver.Vec(dist_ if world > 1 else None)
    V.consistent = {}
    for lev in levels:
        if lev.dm.dot_weight is not None:
            V.set_weight(lev.dm.nglobal, lev.dm.dot_weight)
        V.consistent[lev.dm.nglobal] = lev.dm.make_consistent
    faces = list(app.clamp.keys())
    amg = (RedundantAMG(levels[0].dm, sh.mesh, sh.gmesh, faces, dist_, max_coarse=60) if world > 1 else
           SmoothedAggregationAMG(levels[0].dm, sh.mesh, max_coarse=60))
    pc = solver.PMultigrid(V, levels, transfers, amg=amg)
    U = levels[-1].dm.create_global_vector(matops.MEM_HOST)
    out = solver.newton_solve(V, levels[-1], pc, U, num_increments=app.num_steps)
    return out, U, sh


def _solve_worker(rank, world, port, coarse, out):
    _init(rank, world, port)
    try:
        from oracle_levels import oracle_solve
        app = _app()
        d = dist if world > 1 else None
        if coarse == "amg":
            res, U, sh = _amg_oracle_solve(app, d, rank, world)
            nodes = sh.mesh.node_ids(2) if world > 1 else np.arange(sh.mesh.num_nodes(2))
        else:
            res, U = oracle_solve(app, coarse=coarse, masked=True, dist=d, rank=rank, world=world)
            m = app.mesh
            nodes = m.brick(grid_for(world), rank).node_ids(2) if world > 1 else np.arange(m.num_nodes(2))
        np.savez(os.path.join(out, f"s{coarse}{world}_{rank}.npz"), gdof=_dofs(nodes), u=U.numpy(),
                 snes=res["snes_its"], ksp=res["ksp_its"], conv=res["converged"])
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("coarse", ["pcg", "amg"])
def test_partitioned_newton_krylov_pmg_solve_on_a_tube_matches_serial(tmp_path, coarse):
    """hyperFS p = 2 on a closed tube, oracle operators, 2 gloo ranks against 1: the tolerances of the box test
    (test_halo_gloo.test_partitioned_newton_krylov_pmg_solve_matches_serial)"""
    res = {}
    for world in (1, 2):
        _spawn(_solve_worker, world, coarse, str(tmp_path))
        res[world] = [np.load(tmp_path / f"s{coarse}{world}_{r}.npz") for r in range(world)]
    ser = res[1][0]
    assert bool(ser["conv"])
    us = np.zeros(ser["gdof"].max() + 1)
    us[ser["gdof"]] = ser["u"]
    for d in res[2]:
        assert bool(d["conv"])
        assert int(d["snes"]) == int(ser["snes"])
        assert abs(int(d["ksp"]) - int(ser["ksp"])) <= 0.25 * int(ser["ksp"])
        assert np.linalg.norm(d["u"] - us[d["gdof"]]) < 1e-6 * np.linalg.norm(us)


# --------------------------------------------------------------------------- redundant AMG (gloo)


def _vcycle_mesh(kind):
    """(global mesh, Dirichlet faces): the closed tube, or a box split into bricks"""
    if kind == "box":
        from ceedpetscsolid_b200.mesh import BoxMesh
        return BoxMesh(n=(8, 6, 4), perturb=0.08, seed=0), [(0, 0)]
    return _mesh("tube"), [1]


def _vcycle_worker(rank, world, port, kind, out):
    _init(rank, world, port)
    try:
        from ceedpetscsolid_b200 import matops
        from ceedpetscsolid_b200.amg import RedundantAMG, _global_node_ids
        from amg_helpers import CoarseStub, Coo, oracle_element_matrices
        m, faces = _vcycle_mesh(kind)
        sub = m.brick(grid_for(world), rank, interface_first=True)
        halo = Halo(m, grid_for(world), rank, 1, dist, device="cpu")
        dm = matops.LevelDM(sub, 1, bc_faces=faces, halo=halo, device="cpu", masked=True)
        amg = RedundantAMG(dm, sub, m, faces, dist, max_coarse=30)
        amg.setup(CoarseStub(Coo(sub, oracle_element_matrices(sub))))
        bg = np.random.default_rng(11).standard_normal(m.lsize(1))
        gdof = _dofs(_global_node_ids(sub, m))
        b = torch.from_numpy(bg[gdof].copy())
        dm.zero_constrained(b)
        x = torch.zeros_like(b)
        amg.solve(b, x)
        np.savez(os.path.join(out, f"v{rank}.npz"), gdof=gdof, x=x.numpy(), nlev=len(amg.levels),
                 A=np.concatenate([lev.A.vals.numpy() for lev in amg.levels]))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("kind,world", [("tube", 2), ("box", 4)])
def test_redundant_amg_vcycle_equals_the_one_rank_solve_bit_for_bit(tmp_path, kind, world):
    from ceedpetscsolid_b200 import matops
    from ceedpetscsolid_b200.amg import SmoothedAggregationAMG
    from amg_helpers import CoarseStub, Coo, oracle_element_matrices
    _spawn(_vcycle_worker, world, kind, str(tmp_path))
    m, faces = _vcycle_mesh(kind)
    dm = matops.LevelDM(m, 1, bc_faces=faces, device="cpu", masked=True)
    amg = SmoothedAggregationAMG(dm, m, max_coarse=30)
    amg.setup(CoarseStub(Coo(m, oracle_element_matrices(m))))
    assert len(amg.levels) >= 3
    b = torch.from_numpy(np.random.default_rng(11).standard_normal(m.lsize(1)))
    dm.zero_constrained(b)
    x = torch.zeros_like(b)
    amg.solve(b, x)
    A = np.concatenate([lev.A.vals.numpy() for lev in amg.levels])
    for r in range(world):
        d = np.load(tmp_path / f"v{r}.npz")
        assert int(d["nlev"]) == len(amg.levels)
        assert np.array_equal(d["A"], A), f"rank {r}: hierarchy differs from the one-rank set-up"
        assert np.array_equal(d["x"], x.numpy()[d["gdof"]]), f"rank {r}: V-cycle output differs"


def test_redundant_amg_refuses_the_compressed_layout():
    from ceedpetscsolid_b200.elasticity import AppCtx, Elasticity
    with pytest.raises(NotImplementedError, match="masked layout"):
        Elasticity(AppCtx(n=(4, 4, 4), degree=2), world=2, coarse="amg", masked=False)
