"""Smoothed-aggregation AMG coarse solve (ceedpetscsolid_b200.amg) on the CPU: aggregation, tentative prolongator,
pair-list products against scipy, the Galerkin operator, mesh independence and the whole solve under the oracle."""
import numpy as np
import pytest
import torch

from ceedpetscsolid_b200 import matops, solver
from ceedpetscsolid_b200.amg import (SmoothedAggregationAMG, aggregate, node_graph, rigid_body_modes,
                                     tentative_prolongator)
from ceedpetscsolid_b200.elasticity import AppCtx
from ceedpetscsolid_b200.exodus import HexMesh, tube_mesh
from ceedpetscsolid_b200.mesh import BoxMesh
from amg_helpers import CoarseStub, Coo, amg_oracle_solve, assembled, oracle_element_matrices


def _box_as_hexmesh():
    b = BoxMesh(n=(6, 5, 4), perturb=0.08, seed=0)
    return HexMesh(b.vertices.reshape(-1, 3), b.offsets(1) // 3, {})


def _aggregates(mesh, bc):
    nn = mesh.num_nodes(1)
    free = ~mesh.boundary_mask(1, bc) if bc else np.ones(nn, bool)
    ptr, ind = node_graph(mesh.offsets(1).reshape(-1, 8).astype(np.int64) // 3, nn)
    return free, aggregate(ptr, ind, free)


@pytest.mark.parametrize("which", ["tube", "box"])
def test_aggregation_covers_every_free_node_once_and_is_deterministic(which):
    mesh = tube_mesh(2, 12, 6) if which == "tube" else _box_as_hexmesh()
    bc = [1] if which == "tube" else None
    if which == "box":   # clamp the x = 0 face of the box: constrained nodes by coordinate
        nn = mesh.num_nodes(1)
        free = np.abs(mesh.node_coords(1)[:, 0]) > 1e-12
        ptr, ind = node_graph(mesh.offsets(1).reshape(-1, 8).astype(np.int64) // 3, nn)
        agg, na = aggregate(ptr, ind, free)
        agg2, na2 = aggregate(ptr, ind, free)
    else:
        free, (agg, na) = _aggregates(mesh, bc)
        _, (agg2, na2) = _aggregates(mesh, bc)
    assert (~free).any() and free.any()
    assert np.all(agg[~free] == -1) and np.all(agg[free] >= 0)          # free nodes in one aggregate, constrained in none
    sizes = np.bincount(agg[free], minlength=na)
    assert na > 1 and sizes.min() >= 3 and sizes.sum() == free.sum()
    assert na2 == na and np.array_equal(agg, agg2)


def test_tentative_prolongator_is_orthonormal_and_reproduces_rigid_body_modes():
    mesh = tube_mesh(2, 12, 6)
    free, (agg, na) = _aggregates(mesh, [1])
    X = mesh.node_coords(1)
    center = X[free].mean(axis=0)
    B = rigid_body_modes(X, center)
    Q, R, cen, w = tentative_prolongator(agg, na, B, X, np.ones(X.shape[0]), center)
    fn = np.flatnonzero(free)
    assert np.array_equal(w, np.bincount(agg[fn], minlength=na))
    for a in range(na):
        m = np.flatnonzero(agg[fn] == a)
        q = Q[m].reshape(-1, 6)
        assert np.abs(q.T @ q - np.eye(6)).max() <= 1e-13
        assert np.abs(cen[a] - X[fn[m]].mean(axis=0)).max() < 1e-14
        assert np.abs(q @ R[a] - B[fn[m]].reshape(-1, 6)).max() <= 1e-12 * max(1.0, np.abs(B).max())
    # the global rigid-body modes (rotations about the common centre) on the free nodes: P_tent e_k on every aggregate
    for k in range(6):
        rb = np.eye(3)[k] * np.ones((X.shape[0], 1)) if k < 3 else np.cross(np.eye(3)[k - 3], X - center)
        coarse = R[:, :, k].reshape(-1)
        got = np.einsum("nij,nj->ni", Q, coarse.reshape(na, 6)[agg[fn]])
        assert np.abs(got - rb[fn]).max() < 1e-12 * max(1.0, np.abs(rb).max())


def test_rigid_body_modes_survive_every_level_of_a_floating_patch():
    """the near-null space is carried to every level: the global mode k, written in level-(l+1) coordinates (column k
    of the near-null blocks handed down), is mapped by the level-l tentative and smoothed prolongators onto its level-l
    coordinates, and the Galerkin operator of every coarse level annihilates it"""
    m = tube_mesh(4, 32, 16)
    K = oracle_element_matrices(m)
    dm = matops.LevelDM(m, 1, bc_faces=None, device="cpu", masked=True)
    amg = SmoothedAggregationAMG(dm, m, max_coarse=30)
    with pytest.raises(torch.linalg.LinAlgError):   # no Dirichlet nodes: every level is singular, no Cholesky factor
        amg.setup(CoarseStub(Coo(m, K)))
    assert len(amg.levels) >= 4
    X = m.node_coords(1)
    # scale of the operators: bound on the largest eigenvalue of A_0 (the orthonormal P_tent keep every level near it)
    lam = np.abs(amg.levels[0].A.to_scipy()).sum(axis=1).max()
    for k in range(6):
        rb = np.eye(3)[k] * np.ones((X.shape[0], 1)) if k < 3 else np.cross(np.eye(3)[k - 3], X - amg.center)
        v = rb.reshape(-1)
        for l, lev in enumerate(amg.levels[:-1]):
            c = amg.near_null[l + 1][:, :, k].reshape(-1)
            Pt, P = lev.Pt.to_scipy(), lev.P.to_scipy()
            assert np.abs(Pt @ c - v).max() < 1e-11 * np.abs(v).max(), (k, l)
            assert np.abs(P @ c - v).max() < 1e-8 * np.abs(v).max(), (k, l)
            Ac = amg.levels[l + 1].A.to_scipy()
            assert c @ (Ac @ c) <= 1e-10 * lam * (c @ c), (k, l + 1)
            v = c


def _random_spd_hierarchy(max_coarse=30):
    m = tube_mesh(2, 16, 8)
    dm = matops.LevelDM(m, 1, bc_faces=[1], device="cpu", masked=True)
    E = m.nelem
    rng = np.random.default_rng(5)
    G = rng.standard_normal((E, 24, 24))
    K = np.einsum("eij,ekj->eik", G, G) + 24 * np.eye(24)
    amg = SmoothedAggregationAMG(dm, m, max_coarse=max_coarse)
    amg.setup(CoarseStub(Coo(m, K)))
    return m, dm, K, amg


def _rel(a, b):
    return abs(a - b).max() / max(abs(b).max(), 1e-300)


def test_pair_list_products_equal_scipy():
    m, dm, K, amg = _random_spd_hierarchy()
    assert len(amg.levels) >= 3
    A = assembled(m, K, dm)
    assert _rel(amg.levels[0].A.to_scipy(), A) <= 1e-13
    for l, lev in enumerate(amg.levels[:-1]):
        A = lev.A.to_scipy().tocsr()
        Pt = lev.Pt.to_scipy().tocsr()
        dinv = 1.0 / A.diagonal()
        omega = float(lev.omega[0])
        import scipy.sparse as sp
        assert _rel(lev.P.to_scipy(), Pt - omega * sp.diags(dinv) @ (A @ Pt)) <= 1e-13
        P = lev.P.to_scipy().tocsr()
        assert _rel(lev.PT.to_scipy(), P.T) == 0.0
        assert _rel(lev.AP.to_scipy(), A @ P) <= 1e-13
        assert _rel(amg.levels[l + 1].A.to_scipy(), P.T @ A @ P) <= 1e-13


def test_galerkin_operator_is_spd_and_keeps_exactly_the_rigid_body_null_space():
    m = tube_mesh(2, 12, 4)
    K = oracle_element_matrices(m)
    # clamped end: every level is SPD
    dm = matops.LevelDM(m, 1, bc_faces=[1], device="cpu", masked=True)
    amg = SmoothedAggregationAMG(dm, m, max_coarse=60)
    amg.setup(CoarseStub(Coo(m, K)))
    assert len(amg.levels) >= 2
    for lev in amg.levels[1:]:
        Ac = lev.A.to_scipy().toarray()
        assert np.abs(Ac - Ac.T).max() <= 1e-13 * np.abs(Ac).max()
        assert np.linalg.eigvalsh(Ac).min() > 0
    # free-floating patch: A has the six rigid-body modes as null space, and A_c has those six and nothing else
    dmf = matops.LevelDM(m, 1, bc_faces=None, device="cpu", masked=True)
    amg = SmoothedAggregationAMG(dmf, m, max_coarse=60)
    with pytest.raises(torch.linalg.LinAlgError):   # the coarsest level is singular too: no Cholesky factor
        amg.setup(CoarseStub(Coo(m, K)))
    A = amg.levels[0].A.to_scipy().toarray()
    Ac = amg.levels[1].A.to_scipy().toarray()
    ev, evc = np.linalg.eigvalsh(A), np.linalg.eigvalsh(Ac)
    assert np.sum(ev < 1e-10 * ev.max()) == 6 and np.sum(evc < 1e-10 * evc.max()) == 6
    X = m.node_coords(1)
    P = amg.levels[0].P.to_scipy().toarray()
    for k in range(6):      # coarse representation of the global rigid-body modes: Rayleigh quotient ~ 0
        rb = np.eye(3)[k] * np.ones((X.shape[0], 1)) if k < 3 else np.cross(np.eye(3)[k - 3], X)
        c = np.linalg.lstsq(P, rb.reshape(-1), rcond=None)[0]
        assert np.abs(P @ c - rb.reshape(-1)).max() < 1e-10 * np.abs(rb).max()
        assert c @ Ac @ c <= 1e-12 * evc.max() * (c @ c)


def test_amg_preconditioned_cg_is_mesh_independent_on_the_oracle_operator():
    """linear elasticity on tubes refined in every direction, clamped at one end: CG with one AMG V-cycle stays within
    1.5x of the smallest mesh's count, Jacobi-PCG grows well past that"""
    its_amg, its_jac = [], []
    for nr, nt, nz in [(1, 8, 4), (2, 16, 8), (4, 32, 16)]:
        m = tube_mesh(nr, nt, nz)
        dm = matops.LevelDM(m, 1, bc_faces=[1], device="cpu", masked=True)
        K = oracle_element_matrices(m)
        amg = SmoothedAggregationAMG(dm, m, max_coarse=100)
        amg.setup(CoarseStub(Coo(m, K)))
        assert len(amg.levels) >= 2
        A = assembled(m, K, dm)
        b = torch.from_numpy(np.random.default_rng(0).standard_normal(dm.nglobal))
        dm.zero_constrained(b)
        V = solver.Vec()
        Am = lambda x, y: y.copy_(torch.from_numpy(A @ x.numpy()))
        x = torch.zeros_like(b)
        k, reason, _ = solver.pcg(V, Am, b, x, M=amg.solve, rtol=1e-8, maxit=500)
        assert reason == "rtol"
        assert np.linalg.norm(A @ x.numpy() - b.numpy()) < 1e-6 * np.linalg.norm(b.numpy())
        its_amg.append(k)
        dinv = torch.from_numpy(1.0 / A.diagonal())
        x = torch.zeros_like(b)
        k, reason, _ = solver.pcg(V, Am, b, x, M=lambda r, z: torch.mul(dinv, r, out=z), rtol=1e-8, maxit=5000)
        assert reason == "rtol"
        its_jac.append(k)
    assert max(its_amg) <= 1.5 * its_amg[0], its_amg
    assert its_jac[-1] > 1.5 * its_jac[0] and its_jac[-1] > 1.5 * its_amg[-1], (its_jac, its_amg)


def _tube_app():
    m = tube_mesh(2, 24, 12, r0=0.6, r1=1.0, length=1.5)
    return AppCtx(problem="hyperFS", degree=2, num_steps=2, mesh=m,
                  clamp={1: [0, 0, 0, 0, 0, 1, 0], 2: [0.02, 0, -0.05, 0, 0, 1, 0.05]})


def test_whole_solve_with_amg_converges_to_the_jacobi_pcg_solution():
    """hyperFS p = 2 on a tube whose p = 1 level has two AMG levels.  Measured here: 88 outer CG iterations in 6 Newton
    steps with one V-cycle per coarse solve, 59 with Jacobi-PCG to rtol 1e-2 -- on a two-level hierarchy this small one
    V-cycle is a weaker (but fixed) coarse solve than Jacobi-PCG solved to 1e-2; the bound guards that measured ratio."""
    from oracle_levels import oracle_solve
    ref, Uref = oracle_solve(_tube_app())          # unstructured mesh: Jacobi-PCG coarse solve
    out, U, pc = amg_oracle_solve(_tube_app())
    assert len(pc.amg.levels) >= 2
    assert out["converged"] and ref["converged"]
    assert out["coarse_its"] == out["coarse_solves"] > 0          # one V-cycle per coarse solve
    assert out["snes_its"] == ref["snes_its"] and out["ksp_its"] <= 1.6 * ref["ksp_its"], (out, ref)
    assert np.linalg.norm(U.numpy() - Uref.numpy()) < 1e-6 * np.linalg.norm(Uref.numpy())


def test_amg_coarse_solve_refuses_partitioned_runs():
    from ceedpetscsolid_b200.elasticity import Elasticity
    with pytest.raises(NotImplementedError, match="one GPU"):
        Elasticity(AppCtx(n=(4, 4, 4), degree=2), world=2, coarse="amg")
