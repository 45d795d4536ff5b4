"""Smoothed-aggregation AMG coarse solve on the B200: kernels against their CPU branches, bit-identical set-ups, and
the Newton-Krylov-p-MG solve with coarse='amg' against the oracle harness."""
import numpy as np
import pytest
import torch

from ceedpetscsolid_b200 import matops
from ceedpetscsolid_b200.amg import SmoothedAggregationAMG
from ceedpetscsolid_b200.elasticity import AppCtx
from ceedpetscsolid_b200.exodus import tube_mesh
from amg_helpers import CoarseStub, Coo, amg_oracle_solve

pytestmark = pytest.mark.gpu


def _hierarchy(device, K, m, max_coarse=30):
    dm = matops.LevelDM(m, 1, bc_faces=[1], device=device, masked=True)
    coo = Coo(m, K)
    coo.elem_nodes, coo._v = coo.elem_nodes.to(device), coo._v.to(device)
    amg = SmoothedAggregationAMG(dm, m, max_coarse=max_coarse)
    amg.setup(CoarseStub(coo))
    return amg, coo


def _rel(a, b):
    return float((a.cpu() - b.cpu()).abs().max() / b.abs().max().cpu())


def test_amg_kernels_match_the_cpu_branch_and_are_bit_identical():
    m = tube_mesh(2, 16, 8)
    rng = np.random.default_rng(3)
    G = rng.standard_normal((m.nelem, 24, 24))
    K = np.einsum("eij,ekj->eik", G, G) + 24 * np.eye(24)
    cpu, _ = _hierarchy("cpu", K, m)
    gpu, coo = _hierarchy("cuda", K, m)
    assert len(gpu.levels) == len(cpu.levels) >= 3
    # the lambda_max estimates (and so omega) agree to round-off; the products are compared given the same inputs
    for lc, lg in zip(cpu.levels, gpu.levels):
        assert _rel(lg.A.vals, lc.A.vals) <= 1e-12
    for lc, lg in zip(cpu.levels[:-1], gpu.levels[:-1]):
        for name in ("P", "PT", "AP"):
            assert _rel(getattr(lg, name).vals, getattr(lc, name).vals) <= 1e-12, name
        # products alone, same inputs on both sides: 1e-13
        A, Pt = lg.A.vals, lg.Pt.vals
        for epi in (False, True):
            kw = dict(tmap=lg.tmap, rowof=lg.prow, T=Pt, dinv=lg.sm.dinv, omega=lg.omega) if epi else {}
            out_g = torch.empty_like(lg.P.vals)
            lg.AP_t.run(A, Pt, out_g, **kw)
            kwc = {k: v.cpu() for k, v in kw.items()}
            out_c = torch.empty_like(lc.P.vals)
            lc.AP_t.run(A.cpu(), Pt.cpu(), out_c, **kwc)
            assert _rel(out_g, out_c) <= 1e-13
        out_g = torch.empty_like(lg.AP.vals)
        lg.AP_p.run(A, lg.P.vals, out_g)
        out_c = torch.empty_like(lc.AP.vals)
        lc.AP_p.run(A.cpu(), lg.P.vals.cpu(), out_c)
        assert _rel(out_g, out_c) <= 1e-13
    # SpMV, all four block shapes: (3,3) A0, (3,6) P0, (6,3) P0^T, (6,6) A1
    l0, l1 = gpu.levels[0], gpu.levels[1]
    c0, c1 = cpu.levels[0], cpu.levels[1]
    for Mg, Mc in ((l0.A, c0.A), (l0.P, c0.P), (l0.PT, c0.PT), (l1.A, c1.A)):
        Mc.vals.copy_(Mg.vals.cpu())
        x = torch.from_numpy(rng.standard_normal(Mg.nbcols * Mg.bc))
        yg = torch.zeros(Mg.n, dtype=torch.float64, device="cuda")
        yc = torch.zeros(Mg.n, dtype=torch.float64)
        Mg.mult(x.cuda(), yg)
        Mc.mult(x, yc)
        assert _rel(yg, yc) <= 1e-13, (Mg.br, Mg.bc)
    # a second set-up reproduces every level bit for bit
    before = [lev.A.vals.clone() for lev in gpu.levels] + [gpu.Cinv.vals.clone()]
    gpu.setup(CoarseStub(coo))
    after = [lev.A.vals for lev in gpu.levels] + [gpu.Cinv.vals]
    assert all(torch.equal(a, b) for a, b in zip(before, after))


def _tube_app(steps=2):
    m = tube_mesh(2, 8, 3, r0=0.6, r1=1.0, length=1.0)
    return AppCtx(problem="hyperFS", degree=4, num_steps=steps, mesh=m,
                  clamp={1: [0, 0, 0, 0, 0, 1, 0], 2: [0.02, 0, -0.05, 0, 0, 1, 0.05]})


@pytest.mark.parametrize("deterministic", [False, True])
def test_tube_solve_with_amg_matches_the_oracle_harness(deterministic):
    from ceedpetscsolid_b200.elasticity import Elasticity
    app = _tube_app()
    ref, Uref, pco = amg_oracle_solve(app, max_coarse=60)
    el = Elasticity(_tube_app(), coarse="amg", amg_max_coarse=60, deterministic=deterministic)
    assert el.pc.amg is not None and len(el.pc.amg.levels) == len(pco.amg.levels) >= 2
    out = el.solve()
    assert out["converged"] and ref["converged"]
    assert (out["snes_its"], out["ksp_its"]) == (ref["snes_its"], ref["ksp_its"]), (out, ref)
    assert out["coarse_its"] == out["coarse_solves"]
    u = el.U.cpu().numpy()
    assert np.linalg.norm(u - Uref.numpy()) < 1e-9 * np.linalg.norm(Uref.numpy())


def test_box_solve_with_amg_is_close_to_h_multigrid():
    from ceedpetscsolid_b200.elasticity import Elasticity
    res = {}
    for coarse in ("hmg", "amg"):
        app = AppCtx(problem="hyperFS", degree=4, n=(16, 16, 16), num_steps=2, perturb=0.05)
        el = Elasticity(app, coarse=coarse)
        res[coarse] = el.solve()
        assert res[coarse]["converged"]
        del el
    assert res["amg"]["snes_its"] == res["hmg"]["snes_its"]
    assert res["amg"]["ksp_its"] <= 1.5 * res["hmg"]["ksp_its"], res
