"""K13: CeedOperatorLinearAssemble for JIT-compiled user QFunctions (csrc/b200_jit_assemble.cuh).  The element
matrices of a trilinear level, assembled around the user function, against the oracle's Jacobian column by column,
against the built-in K8 matrices on the same state, and against a host reference built with gcc from the same
header; and user models solved with the assembled coarse level on meshes where probing the operator is refused.
FP64, 1e-12 relative unless stated."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

from ceedpetscsolid_b200 import ceed as libceed
from ceedpetscsolid_b200.ceed import b2, lib
from ceedpetscsolid_b200.exodus import tube_mesh
from helpers import OracleProblem, reoriented, rel_err
from jit_models import EDGE_AI, EDGE_AO, EDGE_CTX, EDGE_FIELDS, EDGE_IN, EDGE_OUT, EXTRA_FIELDS
from oracle import oracle
from test_gpu_jit import SVK_HEADER, _host_point_model, port_locators
from test_gpu_jit_fused import extra_operator

pytestmark = pytest.mark.gpu
TOL = 1e-12


@pytest.fixture
def G():
    assert torch.cuda.is_available()
    import gpu_helpers
    return gpu_helpers


@pytest.fixture
def pair(G, monkeypatch):
    """(K13 problem with the port model of `problem`, built-in problem), both linearised at the same state"""
    from ceedpetscsolid_b200 import setuplibceed

    def make(problem, n, p, resource="/gpu/b200:jit", **kw):
        with monkeypatch.context() as m:
            m.setattr(setuplibceed, "setup_all",
                      functools.partial(setuplibceed.setup_all, qf_locators=port_locators(problem)))
            j = G.GpuProblem(problem, n, p, resource=resource, **kw)
        b = G.GpuProblem(problem, n, p, **kw)
        assert j.data[0].opJacob.is_jit_fused and b.data[0].opJacob.is_fused
        j.residual()
        b.residual()
        return j, b
    return make


def coo(g, level=0):
    """(values, rows, cols) of CeedOperatorLinearAssemble[Symbolic] on the Jacobian of `level`"""
    op = g.data[level].opJacob
    rows, cols = op.linear_assemble_symbolic()
    vals = g.ceed.Vector(rows.size)
    op.linear_assemble(vals)
    v = vals.to_numpy()
    vals.destroy()
    return v, rows, cols


def dense(v, rows, cols, n):
    A = np.zeros((n, n))
    np.add.at(A, (rows, cols), v)
    return A


def close(a, b, tol=TOL):
    return np.max(np.abs(a - b)) <= tol * np.max(np.abs(b))


# ------------------------------------------------------------------------------ 1. the stock models, every (2, Q)
@pytest.mark.parametrize("problem", ["linElas", "hyperSS", "hyperFS"])
@pytest.mark.parametrize("Q", [2, 3, 4, 5])
def test_port_jacobians_are_the_oracle_and_k8_matrices(pair, problem, Q):
    p = Q - 1
    n = (2, 2, 1) if Q > 3 else (3, 2, 2)
    j, b = pair(problem, n, p)
    vj, rows, cols = coo(j)
    vb, rb, cb = coo(b)
    np.testing.assert_array_equal(rows, rb)
    np.testing.assert_array_equal(cols, cb)
    assert close(vj, vb), f"K13 vs K8: {np.abs(vj - vb).max()} of {np.abs(vb).max()}"
    o = OracleProblem(problem, n, p, pl=1)
    A = dense(vj, rows, cols, o.lsize)
    Ao = np.stack([o.jacobian(e) for e in np.eye(o.lsize)], axis=1)
    assert rel_err(A, Ao) < TOL
    if problem != "linElas":
        assert rel_err(A, A.T) < TOL
    assert rel_err(np.diag(A), j.diagonal(0)) < TOL


@pytest.mark.parametrize("count", ["1", "EB-1", "EB", "EB+1", "3EB+2"])
@pytest.mark.parametrize("Q", [3, 5])
def test_group_edges_against_k8(pair, Q, count):
    EB = lib.b200_elems_per_block(Q)
    nelem = {"1": 1, "EB-1": EB - 1, "EB": EB, "EB+1": EB + 1, "3EB+2": 3 * EB + 2}[count]
    j, b = pair("hyperFS", (nelem, 1, 1), Q - 1)
    vj, vb = coo(j)[0], coo(b)[0]
    assert vj.size == 576 * nelem
    assert close(vj, vb), f"{nelem} elements at Q = {Q}"


@pytest.mark.parametrize("p", [2, 4])
def test_a_reoriented_tube_against_k8(pair, p):
    """neighbouring elements with different local axes; 30 elements: a tail group"""
    j, b = pair("hyperFS", None, p, mesh=reoriented(tube_mesh(2, 5, 3), seed=4))
    vj, rows, cols = coo(j)
    vb, rb, cb = coo(b)
    np.testing.assert_array_equal(rows, rb)
    assert close(vj, vb)


# ------------------------------------------------------------------- 2. a model of 8 + 8 fields, active fields 7 and 3
def shape_gradients(Q):
    """G[q][node][k]: reference gradients of the trilinear shape functions, q = qx + Q qy + Q^2 qz"""
    B, D = (np.asarray(m) for m in oracle.basis_1d(2, Q, 0)[:2])
    G = np.zeros((Q ** 3, 8, 3))
    for q in range(Q ** 3):
        qx, qy, qz = q % Q, (q // Q) % Q, q // (Q * Q)
        for i in range(8):
            ix, iy, iz = i & 1, (i >> 1) & 1, i >> 2
            G[q, i] = (D[qx, ix] * B[qy, iy] * B[qz, iz], B[qx, ix] * D[qy, iy] * B[qz, iz],
                       B[qx, ix] * B[qy, iy] * D[qz, iz])
    return B, D, G


def element_matrices(Dt, Q):
    """K[e][col = j*3 + b][row = i*3 + a] = sum_q sum_{k,m} G[q,i,k] Dt[e,q,m*3 + b,k*3 + a] G[q,j,m], flattened to
    [e][576]: the trilinear element matrices of a point tangent Dt[e][q][s][o] (test_gpu_jit_diag.host_tangent's
    layout)"""
    nelem, nq = Dt.shape[:2]
    _, _, Gs = shape_gradients(Q)
    Dr = Dt.reshape(nelem, nq, 3, 3, 3, 3)                 # [e][q][m][b][k][a]
    return np.einsum("qik,eqmbka,qjm->ejbia", Gs, Dr, Gs).reshape(nelem, 576)


def qblocked(a):
    """[elem][comp][q] -> the q-blocked backend layout"""
    from test_gpu_operator_kernels import to_qb
    return to_qb(a)


@pytest.mark.parametrize("Q", [2, 3, 5])
def test_edge_model_against_its_host_tangent(tmp_path, Q):
    nelem = 2 * lib.b200_elems_per_block(Q) + 1
    nq = Q ** 3
    (tmp_path / "edge.h").write_text(EDGE_FIELDS)
    rng = np.random.default_rng(Q)
    pin = [rng.uniform(-1, 1, (nelem, w, nq)) for w in EDGE_IN[:EDGE_AI]]
    k = rng.uniform(-1, 1, EDGE_CTX)
    k[255] = 0.0                      # the active output is then linear in the active input
    ctx = (C.c_double * EDGE_CTX)(*k)
    # host tangent: the gcc build of EdgeF at the 9 unit active inputs
    Dt = np.zeros((nelem, nq, 9, 9))  # [e][q][s][o]
    for s in range(9):
        act = np.zeros((nelem, 9, nq))
        act[:, s, :] = 1.0
        sub = tmp_path / f"host{s}"
        sub.mkdir()
        (sub / "edge.h").write_text(EDGE_FIELDS)
        outs = _host_point_model(sub, ctx, nelem, nq, pin + [act], EDGE_OUT, header="edge.h", name="EdgeF")
        Dt[:, :, s, :] = outs[EDGE_AO].transpose(0, 2, 1)
    B, D, _ = shape_gradients(Q)
    ref = element_matrices(Dt, Q)
    h = libceed.jit_assemble_compile(tmp_path / "edge.h", "EdgeF", EDGE_IN, EDGE_OUT, EDGE_AI, EDGE_AO, 2, Q)
    d_in = [torch.from_numpy(qblocked(a)).cuda() for a in pin]
    ptrs = [t.data_ptr() for t in d_in] + [0]
    vals = torch.full((nelem * 576,), np.nan, dtype=torch.float64, device="cuda")
    Bc, Dc = np.ascontiguousarray(B), np.ascontiguousarray(D)
    b2(lib.b200_jit_assemble_apply(h, C.addressof(ctx), C.sizeof(ctx), nelem, Bc.ctypes.data, Dc.ctypes.data, 8,
                                   (C.c_void_p * 8)(*ptrs), vals.data_ptr()))
    torch.cuda.synchronize()
    got = vals.cpu().numpy().reshape(nelem, 576)
    assert close(got, ref), np.abs(got - ref).max()


# ------------------------------------------------------------------------------------------- 3. semantics, refusals
def test_passive_outputs_are_untouched_by_assembly(G, tmp_path):
    """ExtraF (active fields 1 and 1, passive outputs sdiag and energy): an apply fills the passive outputs, an
    assembly leaves them bitwise as they were"""
    path = tmp_path / "extra.h"
    path.write_text(EXTRA_FIELDS)
    g = G.GpuProblem("linElas", (3, 2, 2), 1, resource="/gpu/b200:jit")
    nelem, nq = g.mesh.nelem, 8
    rng = np.random.default_rng(2)
    qd = np.tile(np.r_[0.125, 2, 0, 0, 0, 2, 0, 0, 0, 2][None, :, None], (nelem, 1, nq))
    op, out = extra_operator(g, path, True, rng.uniform(0, 1, (nelem, 1, nq)), qd)
    assert op.is_jit_fused
    n = g.mesh.lsize(1)
    g.apply(op, rng.standard_normal(n), n)
    before = {name: out(name).copy() for name in ("sdiag", "energy")}
    assert all(np.isfinite(v).all() for v in before.values())
    rows, cols = op.linear_assemble_symbolic()
    vals = g.ceed.Vector(rows.size)
    op.linear_assemble(vals)
    assert np.isfinite(vals.to_numpy()).all()
    for name, v in before.items():
        np.testing.assert_array_equal(out(name).view(np.uint64), v.view(np.uint64), err_msg=name)


@pytest.mark.parametrize("resource", ["/gpu/b200:jit", "/gpu/b200:deterministic:jit"])
def test_two_assemblies_are_bitwise_equal(pair, resource):
    j, _ = pair("hyperFS", (5, 3, 2), 4, resource=resource)
    v1, v2 = coo(j)[0], coo(j)[0]
    np.testing.assert_array_equal(v1.view(np.uint64), v2.view(np.uint64))


def test_the_program_compiles_at_the_first_assemble_only(pair, tmp_path):
    j, _ = pair("hyperSS", (3, 2, 2), 3)
    n0 = libceed.jit_compile_count()
    coo(j)
    n1 = libceed.jit_compile_count()
    coo(j)
    assert n1 - n0 <= 1 and libceed.jit_compile_count() == n1   # once per process (0 if an earlier test compiled it)


def test_generic_path_and_other_levels_are_refused(pair, G, monkeypatch):
    from ceedpetscsolid_b200 import setuplibceed
    j, _ = pair("hyperFS", 2, 2)
    with pytest.raises(libceed.CeedError, match=r"trilinear \(P = 2\) level only \(operator port_HyperFSdF, P = 3\)"):
        j.data[1].opJacob.linear_assemble_symbolic()
    with monkeypatch.context() as m:  # qextra = 1 at p = 4: (P, Q) = (2, 6) on the p = 1 level, no fused kernel
        m.setattr(setuplibceed, "setup_all", functools.partial(setuplibceed.setup_all,
                                                               qf_locators=port_locators("hyperFS")))
        g = G.GpuProblem("hyperFS", 2, 4, qextra=1, resource="/gpu/b200:jit")
    assert not g.data[0].opJacob.is_jit_fused
    with pytest.raises(libceed.CeedError, match=r"JIT QFunction port_HyperFSdF runs on the generic path.*\(2, 6\)"):
        g.data[0].opJacob.linear_assemble_symbolic()


# --------------------------------------------------------------------------- 4. solves above the probing limit
TUBE = (4, 32, 48)   # 23 520 p = 1 dofs: column probing refuses it


def _solve(locs, coarse, mesh=None):
    from ceedpetscsolid_b200.elasticity import AppCtx, Elasticity
    if mesh is not None:
        app = AppCtx(problem="hyperFS", degree=2, num_steps=2, mesh=mesh,
                     clamp={1: [0, 0, 0, 0, 0, 1, 0], 2: [0, -0.02, 0.04, 0, 0, 1, 0]})
    else:
        app = AppCtx(problem="hyperFS", degree=2, n=(6, 6, 6), num_steps=2, perturb=0.05)
    el = Elasticity(app, qf_locators=locs, coarse=coarse)
    return el, el.solve()


@pytest.mark.parametrize("coarse", ["pcg", "amg"])
def test_port_model_solves_an_unstructured_tube_like_the_builtin(G, coarse):
    mesh = tube_mesh(*TUBE)
    assert 3 * mesh.num_nodes(1) > 20000
    jel, jout = _solve(port_locators("hyperFS"), coarse, mesh)
    assert jel.users[0].op.is_jit_fused and jel.levels[0].coo is not None
    bel, bout = _solve(None, coarse, mesh)
    assert jout["converged"] and bout["converged"]
    assert (jout["snes_its"], jout["ksp_its"]) == (bout["snes_its"], bout["ksp_its"])
    assert rel_err(jel.U.cpu().numpy(), bel.U.cpu().numpy()) < 1e-9


def test_port_model_amg_on_a_box_like_the_builtin(G):
    jel, jout = _solve(port_locators("hyperFS"), "amg")
    assert jel.levels[0].coo is not None
    bel, bout = _solve(None, "amg")
    assert jout["converged"] and bout["converged"]
    assert (jout["snes_its"], jout["ksp_its"]) == (bout["snes_its"], bout["ksp_its"])
    assert rel_err(jel.U.cpu().numpy(), bel.U.cpu().numpy()) < 1e-9


@pytest.mark.parametrize("coarse", ["pcg", "amg"])
def test_a_model_the_backend_does_not_have_solves_the_tube(G, tmp_path, coarse):
    h = tmp_path / "svk.h"
    h.write_text(SVK_HEADER)
    el, out = _solve({"apply": f"{h}:SvkF", "jacob": f"{h}:SvkdF"}, coarse, tube_mesh(*TUBE))
    assert el.levels[0].coo is not None
    assert out["converged"] and out["snes_its"] >= 2
