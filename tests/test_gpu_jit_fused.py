"""K12: the fused operator kernel generated around a JIT-compiled user QFunction ("/gpu/b200:jit").  Eligible operators
run in one launch (gather, sum-factorised gradient, the user function per point, transposed stages, scatter); the
generic path (restriction, basis, K11 point kernel, transposes) is the reference, with the float64 oracle."""
import functools
import os

import numpy as np
import pytest
import torch

from helpers import OracleProblem, rel_err
from jit_models import EXTRA_FIELDS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
QF_PORT = os.path.join(ROOT, "oracle", "qf_port.c")
TOL = 1e-12
pytestmark = pytest.mark.gpu


def port_locators(problem):
    model = {"linElas": "LinElas", "hyperSS": "HyperSS", "hyperFS": "HyperFS"}[problem]
    return {"apply": f"{QF_PORT}:port_{model}F", "jacob": f"{QF_PORT}:port_{model}dF"}


@pytest.fixture
def G():
    assert torch.cuda.is_available()
    import gpu_helpers
    return gpu_helpers


@pytest.fixture
def jit_problem(G, monkeypatch):
    """GpuProblem whose set-up passes qf_locators to setuplibceed.setup_all"""
    from ceedpetscsolid_b200 import setuplibceed

    def make(problem, n, p, qf_locators, resource="/gpu/b200:jit", **kw):
        with monkeypatch.context() as m:
            m.setattr(setuplibceed, "setup_all", functools.partial(setuplibceed.setup_all, qf_locators=qf_locators))
            return G.GpuProblem(problem, n, p, resource=resource, **kw)
    return make


def qblocked_index(nelem, ncomp, Q):
    """index[e, c, q] of the q-blocked CEED_STRIDES_BACKEND layout (include/b200_kernels.h)"""
    EB, T = (16 if Q <= 3 else 4), Q * Q
    e = np.arange(nelem)[:, None, None]
    c = np.arange(ncomp)[None, :, None]
    q = np.arange(Q ** 3)[None, None, :]
    g = e // EB
    ebn = np.minimum(nelem - g * EB, EB)
    return g * EB * ncomp * Q ** 3 + (c * Q + q % Q) * (ebn * T) + (q // Q) * ebn + (e - g * EB)


# ------------------------------------------------------------------------------------------------ which operators
@pytest.mark.parametrize("problem,n,p", [("linElas", 3, 2), ("hyperSS", 2, 3), ("hyperFS", 2, 4)])
def test_stock_shapes_run_on_k12_at_every_level(jit_problem, problem, n, p):
    g = jit_problem(problem, n, p, port_locators(problem))
    assert g.fine.opApply.is_jit_fused and not g.fine.opApply.is_fused
    for d in g.data:
        assert d.opJacob.is_jit_fused and not d.opJacob.is_fused


def test_shapes_outside_the_table_and_point_operators_stay_generic(jit_problem):
    from ceedpetscsolid_b200 import ceed as libceed
    from ceedpetscsolid_b200.ceed import BASIS_COLLOCATED, EVAL_NONE, VECTOR_ACTIVE
    g = jit_problem("hyperFS", 2, 4, port_locators("hyperFS"), qextra=1)    # Q = 6: (P, Q) = (5, 6), (3, 6), (2, 6)
    assert not g.fine.opApply.is_jit_fused and not any(d.opJacob.is_jit_fused for d in g.data)
    o = OracleProblem("hyperFS", 2, 4, qextra=1)
    assert rel_err(g.residual(), o.residual_fine(o.u_fine)) < TOL
    # a point-only operator: every field EVAL_NONE
    nelem, nq = g.mesh.nelem, 27
    qf = g.ceed.QFunction(1, f"{QF_PORT}:port_LinElasdF")
    for name, s in (("du", 9), ("qdata", 10)):
        qf.add_input(name, s, EVAL_NONE)
    qf.add_output("dv", 9, EVAL_NONE)
    qf.set_context(g.phys)
    op = g.ceed.Operator(qf)
    for name, s in (("du", 9), ("qdata", 10), ("dv", 9)):
        r = g.ceed.StridedElemRestriction(nelem, nq, s, nelem * s * nq)
        v = VECTOR_ACTIVE if name != "qdata" else g.ceed.Vector(nelem * s * nq)
        op.set_field(name, r, BASIS_COLLOCATED, v)
    assert not op.is_jit_fused and not op.is_fused
    assert libceed.jit_compile_count() > 0


# ------------------------------------------------------------------------------------ the generic path as reference
def extra_operator(g, path, blocked, scale, qd_plain):
    """ExtraF (tests/jit_models.py) on g's fine level; passive fields on q-blocked CEED_STRIDES_BACKEND restrictions
    (K12), or on explicit [1, nq, ncomp nq] strides with the data re-laid (generic path)"""
    from ceedpetscsolid_b200 import ceed as libceed
    from ceedpetscsolid_b200.ceed import BASIS_COLLOCATED, EVAL_GRAD, EVAL_NONE, VECTOR_ACTIVE
    d, ceed, nelem = g.fine, g.ceed, g.mesh.nelem
    Q = g.p + 1 + g.qextra
    nq = Q ** 3
    qf = ceed.QFunction(1, f"{path}:ExtraF")
    qf.add_input("scale", 1, EVAL_NONE)
    qf.add_input("du", 9, EVAL_GRAD)
    qf.add_input("qdata", 10, EVAL_NONE)
    qf.add_output("sdiag", 3, EVAL_NONE)
    qf.add_output("dv", 9, EVAL_GRAD)
    qf.add_output("energy", 1, EVAL_NONE)
    qf.set_context(g.phys)
    op = ceed.Operator(qf)
    passive = {}
    for name, nc, data in (("scale", 1, scale), ("qdata", 10, qd_plain), ("sdiag", 3, None), ("energy", 1, None)):
        size = nelem * nc * nq
        if blocked:
            r = ceed.StridedElemRestriction(nelem, nq, nc, size)
            arr = np.full(size, np.nan)
            if data is not None:
                arr[qblocked_index(nelem, nc, Q)] = data
        else:
            r = ceed.StridedElemRestriction(nelem, nq, nc, size, strides=[1, nq, nc * nq])
            arr = data.reshape(-1).copy() if data is not None else np.full(size, np.nan)
        v = ceed.Vector(size)
        v.set_array(arr, libceed.MEM_HOST, libceed.COPY_VALUES)
        passive[name] = (r, v, nc)
    op.set_field("scale", passive["scale"][0], BASIS_COLLOCATED, passive["scale"][1])
    op.set_field("du", d.Erestrictu, d.basisu, VECTOR_ACTIVE)
    op.set_field("qdata", passive["qdata"][0], BASIS_COLLOCATED, passive["qdata"][1])
    op.set_field("sdiag", passive["sdiag"][0], BASIS_COLLOCATED, passive["sdiag"][1])
    op.set_field("dv", d.Erestrictu, d.basisu, VECTOR_ACTIVE)
    op.set_field("energy", passive["energy"][0], BASIS_COLLOCATED, passive["energy"][1])

    def out(name):
        _, v, nc = passive[name]
        a = v.to_numpy()
        return a[qblocked_index(nelem, nc, Q)] if blocked else a.reshape(nelem, nc, nq)
    return op, out


def close(a, b, tol=1e-13):
    return np.max(np.abs(a - b)) <= tol * np.max(np.abs(b))


@pytest.mark.parametrize("p,n", [(4, (3, 3, 3)), (2, (3, 3, 3)), (3, (5, 3, 2))])
def test_extra_passive_fields_against_the_generic_path(G, tmp_path, p, n):
    """27 elements: a tail group of 3 (EB = 4, Q = 5) and of 11 (EB = 16, Q = 3); 30 elements at Q = 4: tail of 2"""
    from ceedpetscsolid_b200 import ceed as libceed
    (tmp_path / "extra.h").write_text(EXTRA_FIELDS)
    g = G.GpuProblem("linElas", n, p, resource="/gpu/b200:jit", multigrid="none")
    nelem, Q = g.mesh.nelem, p + 1
    qd_plain = g.strided_to_plain(g.fine.Erestrictqdi, g.fine.qdata)
    rng = np.random.default_rng(p)
    scale = rng.uniform(0.0, 1.0, (nelem, 1, Q ** 3))
    x = rng.standard_normal(g.mesh.lsize(p))
    res = {}
    for blocked in (True, False):
        op, out = extra_operator(g, tmp_path / "extra.h", blocked, scale, qd_plain)
        assert op.is_jit_fused == blocked and not op.is_fused
        xd = torch.from_numpy(x).cuda()
        y = torch.zeros_like(xd)
        xc, yc = g.ceed.Vector(x.size), g.ceed.Vector(x.size)
        xc.set_array(xd)
        yc.set_array(y)
        op.apply(xc, yc)                       # Apply: passive outputs overwritten (they start as NaN)
        torch.cuda.synchronize()
        first = (y.cpu().numpy(), out("sdiag"), out("energy"))
        op.apply_add(xc, yc)                   # ApplyAdd: added to, active and passive
        torch.cuda.synchronize()
        second = (y.cpu().numpy(), out("sdiag"), out("energy"))
        xc.take_array()
        yc.take_array()
        res[blocked] = first, second
    for k in range(2):
        for i, what in enumerate(("dv", "sdiag", "energy")):
            assert close(res[True][k][i], res[False][k][i]), (k, what)
            assert not np.isnan(res[True][k][i]).any()
    assert close(res[True][1][1], 2 * res[True][0][1])
    assert libceed.jit_compile_count() > 0


# --------------------------------------------------------------------------------------------- stock models, oracle
@pytest.mark.parametrize("problem,n,p", [("linElas", 3, 2), ("hyperSS", 3, 3), ("hyperFS", 3, 4)])
def test_stock_models_on_k12_against_the_oracle(jit_problem, problem, n, p):
    g = jit_problem(problem, n, p, port_locators(problem))
    o = OracleProblem(problem, n, p)
    assert g.fine.opApply.is_jit_fused
    if o.has_gradu:
        g.fine.gradu.set_value(float("nan"))
    assert rel_err(g.residual(), o.residual_fine(o.u_fine)) < TOL
    if o.has_gradu:
        assert rel_err(g.strided_to_plain(g.fine.ErestrictGradui, g.fine.gradu), o.gradu) < TOL
    rng = np.random.default_rng(7)
    for level, deg in enumerate(g.degrees):
        assert g.data[level].opJacob.is_jit_fused
        ol = OracleProblem(problem, n, p, pl=deg)
        x = rng.standard_normal(ol.lsize)
        assert rel_err(g.jacobian(level, x), ol.jacobian(x)) < TOL, level


# --------------------------------------------------------------------------------------------------- determinism
def test_deterministic_k12_is_bit_identical_and_close_to_atomics(jit_problem):
    gd = jit_problem("hyperFS", 3, 4, port_locators("hyperFS"), resource="/gpu/b200:jit:deterministic")
    ga = jit_problem("hyperFS", 3, 4, port_locators("hyperFS"))
    assert gd.ceed.is_deterministic and gd.fine.opJacob.is_jit_fused
    r1, r2, ra = gd.residual(), gd.residual(), ga.residual()
    assert np.array_equal(r1, r2) and close(r1, ra)
    fine = len(gd.degrees) - 1
    x = np.random.default_rng(2).standard_normal(gd.mesh.lsize(4))
    y1, y2, ya = gd.jacobian(fine, x), gd.jacobian(fine, x), ga.jacobian(fine, x)
    assert np.array_equal(y1, y2) and close(y1, ya)


# ------------------------------------------------------------------------------------------------- element ranges
def test_apply_add_range_equals_the_full_apply(jit_problem):
    from ceedpetscsolid_b200 import ceed as libceed
    g = jit_problem("hyperFS", 3, 4, port_locators("hyperFS"))     # 27 elements, EB = 4
    g.residual()
    fine = len(g.degrees) - 1
    op = g.data[fine].opJacob
    x = torch.from_numpy(np.random.default_rng(3).standard_normal(g.mesh.lsize(4))).cuda()
    yf, yr = torch.zeros_like(x), torch.zeros_like(x)
    xc, yc = g.ceed.Vector(x.numel()), g.ceed.Vector(x.numel())
    xc.set_array(x)
    yc.set_array(yf)
    op.apply(xc, yc)
    yc.take_array()
    yc.set_array(yr)
    op.apply_add_range(xc, yc, 0, 12)
    op.apply_add_range(xc, yc, 12, 27)
    with pytest.raises(libceed.CeedError, match="bad element range"):
        op.apply_add_range(xc, yc, 5, 27)
    xc.take_array()
    yc.take_array()
    torch.cuda.synchronize()
    assert close(yr.cpu().numpy(), yf.cpu().numpy(), 1e-14)


# ------------------------------------------------------------------------------------------------ compilations
def test_fused_programs_compile_once_at_first_apply(jit_problem, tmp_path):
    from ceedpetscsolid_b200 import ceed as libceed
    src = tmp_path / "qf_port_copy.c"   # a path of its own: programs this process has not compiled yet
    src.write_text(open(QF_PORT).read())
    n0 = libceed.jit_compile_count()
    g = jit_problem("hyperFS", 2, 4, {"apply": f"{src}:port_HyperFSF", "jacob": f"{src}:port_HyperFSdF"})
    assert g.fine.opApply.is_jit_fused and all(d.opJacob.is_jit_fused for d in g.data)
    assert libceed.jit_compile_count() - n0 == 2   # set-up: the point programs only
    rng = np.random.default_rng(4)
    for rep in range(2):
        g.residual()
        for level, deg in enumerate(g.degrees):
            g.jacobian(level, rng.standard_normal(g.mesh.lsize(deg)))
        # residual (5, 5); Jacobian (2, 5), (3, 5), (5, 5): once each, at the first apply
        assert libceed.jit_compile_count() - n0 == 2 + 1 + 3, rep


# --------------------------------------------------------------------------------------------- partitioned apply
@pytest.mark.parametrize("name", ["box2", "box8"])
def test_partitioned_k12_loopback(jit_problem, monkeypatch, name):
    """the residual and Jacobian of a K12 operator through CeedOperatorApplyPartitionedB200 on loopback bricks
    (tests/test_gpu_halo_loopback.py), every rank in turn with an overlapped split, against the oracle and against the
    one-rank K12 apply of the whole mesh"""
    import test_gpu_halo_loopback as L
    from ceedpetscsolid_b200 import setuplibceed
    problem, p = "hyperFS", 2
    o, gbc = L.oracle_for(name, problem, p)
    _, _, n = L.op_global(name)
    one = jit_problem(problem, n, p, port_locators(problem), multigrid="none")
    monkeypatch.setattr(setuplibceed, "setup_all",
                        functools.partial(setuplibceed.setup_all, qf_locators=port_locators(problem)))
    gmesh, ranks = L.op_ranks(name, problem, p, "/gpu/b200:jit")
    assert all(rk.data.opApply.is_jit_fused and rk.data.opJacob.is_jit_fused for rk in ranks)
    assert all(0 < rk.mesh.n_interface < rk.mesh.nelem for rk in ranks)
    rres = o.residual_fine(o.u_fine)
    r1 = one.residual()
    xg = np.random.default_rng(1).standard_normal(gbc.size)
    xg[gbc] = 0.0
    yjac, y1 = o.jacobian(xg), one.jacobian(0, xg)
    for rk in ranks:
        rk.X.copy_(torch.from_numpy(xg[rk.gdof]))
    with L.Loopback([rk.halo for rk in ranks]) as lb:
        for subject in L.subjects(ranks):
            rk = ranks[subject]
            L.run_subject(ranks, subject, lambda rk: rk.data.opApply, lambda rk: rk.u, rk.mesh.n_interface)
            lb.check()
            outs = [q.Y.cpu().numpy() for q in ranks]
            L.check_against_oracle(ranks, outs, rres, gbc, f"K12 partitioned residual on rank {subject}")
            L.check_against_oracle(ranks, outs, r1, gbc, f"K12 partitioned residual on rank {subject} vs one rank")
            L.run_subject(ranks, subject, lambda rk: rk.data.opJacob, lambda rk: rk.X, rk.mesh.n_interface)
            lb.check()
            outs = [q.Y.cpu().numpy() for q in ranks]
            L.check_against_oracle(ranks, outs, yjac, gbc, f"K12 partitioned Jacobian on rank {subject}")
            L.check_against_oracle(ranks, outs, y1, gbc, f"K12 partitioned Jacobian on rank {subject} vs one rank")
