"""K14: CeedOperatorLinearAssembleDiagonal for JIT-compiled user QFunctions on K12 (csrc/b200_jit_diag.cuh).  The
diagonal, computed around the user function, against the oracle, against the built-in diagonal (K3) on the same
state, against the diagonal of dense matrices probed through K12 applies, and against host tangents built with gcc from
the same header; and user models solved with the Jacobi/Chebyshev smoothers that call it.  FP64, 1e-12 relative
unless stated."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

from ceedpetscsolid_b200 import ceed as libceed
from ceedpetscsolid_b200.ceed import b2, lib
from ceedpetscsolid_b200.exodus import tube_mesh
from helpers import OracleProblem, reoriented, rel_err
from jit_models import EDGE_AI, EDGE_AO, EDGE_CTX, EDGE_FIELDS, EDGE_IN, EDGE_OUT, EXTRA_FIELDS, NONSYM
from oracle import oracle
from test_gpu_jit import SVK_HEADER, _host_point_model, port_locators
from test_gpu_jit_assemble import coo, dense, qblocked
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
    """(K14 problem with the port model of `problem`, built-in problem), both linearised at the same state"""
    from ceedpetscsolid_b200 import setuplibceed

    def make(problem, n, p, resource="/gpu/b200:jit", locators=None, **kw):
        with monkeypatch.context() as m:
            m.setattr(setuplibceed, "setup_all",
                      functools.partial(setuplibceed.setup_all, qf_locators=locators or port_locators(problem)))
            j = G.GpuProblem(problem, n, p, resource=resource, **kw)
        b = G.GpuProblem(problem, n, p, **kw)
        assert all(d.opJacob.is_jit_fused for d in j.data) and all(d.opJacob.is_fused for d in b.data)
        j.residual()
        b.residual()
        return j, b
    return make


def op_diagonal(g, op, n):
    d = torch.zeros(n, dtype=torch.float64, device="cuda")
    dc = g.ceed.Vector(n)
    dc.set_array(d)
    op.linear_assemble_diagonal(dc)
    dc.take_array()
    dc.destroy()
    torch.cuda.synchronize()
    return d.cpu().numpy()


def probed_diagonal(g, op, n):
    """diag of the dense operator, column by column through K12 applies"""
    return np.array([g.apply(op, e, n)[i] for i, e in enumerate(np.eye(n))])


def close(a, b, tol=TOL):
    return np.max(np.abs(a - b)) <= tol * np.max(np.abs(b))


# ------------------------------------------------------------------------------------------------------ 1. routing
def test_first_diagonal_compiles_one_program_per_level(pair, tmp_path):
    src = tmp_path / "qf_port_copy.c"     # a path of its own: programs this process has not compiled yet
    src.write_text(open(port_locators("hyperFS")["jacob"].rsplit(":", 1)[0]).read())
    j, _ = pair("hyperFS", 2, 4, locators={"apply": f"{src}:port_HyperFSF", "jacob": f"{src}:port_HyperFSdF"})
    assert j.degrees == [1, 2, 4]
    for level in range(3):
        n0 = libceed.jit_compile_count()
        j.diagonal(level)
        assert libceed.jit_compile_count() == n0 + 1, level
    n0 = libceed.jit_compile_count()
    for level in range(3):
        j.diagonal(level)
    assert libceed.jit_compile_count() == n0


# ------------------------------------------------------------------------------ 2. the stock models, every (P, Q)
@pytest.mark.parametrize("problem", ["linElas", "hyperSS", "hyperFS"])
@pytest.mark.parametrize("Q", [2, 3, 4, 5])
def test_port_jacobians_are_the_oracle_and_k3_diagonals(pair, problem, Q):
    """uniform p-multigrid at p = Q - 1: levels P = 2..Q, every (P, Q) of B200_FOR_PQ over the four Q"""
    p = Q - 1
    n = (2, 2, 1) if Q > 3 else (3, 2, 2)
    j, b = pair(problem, n, p, multigrid="uniform")
    for level, deg in enumerate(j.degrees):
        dj = j.diagonal(level)
        assert rel_err(dj, OracleProblem(problem, n, p, pl=deg).diagonal()) < TOL, (deg + 1, Q)
        assert rel_err(dj, b.diagonal(level)) < TOL, (deg + 1, Q)


@pytest.mark.parametrize("count", ["1", "EB-1", "EB", "EB+1", "3EB+2"])
@pytest.mark.parametrize("Q", [3, 5])
def test_group_edges_against_k3(pair, Q, count):
    EB = lib.b200_elems_per_block(Q)
    nelem = {"1": 1, "EB-1": EB - 1, "EB": EB, "EB+1": EB + 1, "3EB+2": 3 * EB + 2}[count]
    j, b = pair("hyperFS", (nelem, 1, 1), Q - 1)
    for level in range(len(j.degrees)):
        assert rel_err(j.diagonal(level), b.diagonal(level)) < TOL, (nelem, level)


@pytest.mark.parametrize("p", [2, 4])
def test_a_reoriented_tube_against_k3(pair, p):
    """neighbouring elements with different local axes; 30 elements: a tail group"""
    j, b = pair("hyperFS", None, p, mesh=reoriented(tube_mesh(2, 5, 3), seed=4))
    for level in range(len(j.degrees)):
        assert rel_err(j.diagonal(level), b.diagonal(level)) < TOL, level


def test_a_smoother_context_gives_the_diagonal_for_its_constants(pair):
    """GetDiag_Ceed swaps the Jacobian context for the smoother's; the context is read at every diagonal"""
    j, _ = pair("hyperFS", 2, 2)
    o = OracleProblem("hyperFS", 2, 2)
    fine = len(j.degrees) - 1
    d0 = j.diagonal(fine)
    assert rel_err(d0, o.diagonal()) < TOL
    j.phys.nu, j.phys.E = 0.25, 3.0
    want = oracle.operator_diagonal("hyperFS", (0.25, 3.0), o.nelem, o.P, o.Q, o.B, o.D, o.offsets, o.qdata, o.gradu,
                                    o.lsize, o.which)
    d1 = j.diagonal(fine)
    assert rel_err(d1, want) < TOL
    assert rel_err(d1, d0) > 1e-3


# ------------------------------------------------------------------- 3. a non-symmetric linear model, host tangents
# NONSYM (tests/jit_models.py): a linear model whose point tangent is not symmetric
def shape_gradients(P, Q):
    """G[q][node][k]: reference gradients of the tensor shape functions, q = qx + Q qy + Q^2 qz, node = ix + P iy +
    P^2 iz"""
    B, D = (np.asarray(m) for m in oracle.basis_1d(P, Q, 0)[:2])
    q = np.arange(Q ** 3)
    n = np.arange(P ** 3)
    qx, qy, qz = q % Q, (q // Q) % Q, q // (Q * Q)
    ix, iy, iz = n % P, (n // P) % P, n // (P * P)
    Bx, By, Bz = B[np.ix_(qx, ix)], B[np.ix_(qy, iy)], B[np.ix_(qz, iz)]
    Dx, Dy, Dz = D[np.ix_(qx, ix)], D[np.ix_(qy, iy)], D[np.ix_(qz, iz)]
    return B, D, np.stack([Dx * By * Bz, Bx * Dy * Bz, Bx * By * Dz], axis=-1)


def host_tangent(tmp_path, header, name, ctx, nelem, nq, passive, ai, ao, out_sizes):
    """Dt[e][q][s = m*3 + b][o = k*3 + a] = dW[a][k] / dH[b][m]: the gcc build of `header` at the 9 unit active inputs
    (passive inputs [elem][comp][q], inserted around the active input at index ai)"""
    Dt = np.zeros((nelem, nq, 9, 9))
    for s in range(9):
        act = np.zeros((nelem, 9, nq))
        act[:, s, :] = 1.0
        sub = tmp_path / f"host{s}"
        sub.mkdir()
        (sub / header).write_text((tmp_path / header).read_text())
        outs = _host_point_model(sub, ctx, nelem, nq, passive[:ai] + [act] + passive[ai:], out_sizes, header=header,
                                 name=name)
        Dt[:, :, s, :] = outs[ao].transpose(0, 2, 1)
    return Dt


def element_diagonal(Dt, P, Q):
    """diag_e[e][node][c] = sum_q sum_{k,m} G_k D[c k][c m] G_m of a host tangent Dt (host_tangent's layout)"""
    nelem, nq = Dt.shape[:2]
    Dc = np.einsum("eqmckc->eqmkc", Dt.reshape(nelem, nq, 3, 3, 3, 3))   # D[c k][c m] as [e][q][m][k][c]
    _, _, Gs = shape_gradients(P, Q)
    return np.einsum("qnk,eqmkc,qnm->enc", Gs, Dc, Gs)


def host_element_diagonal(tmp_path, header, name, ctx, nelem, nq, passive, ai, ao, out_sizes, P, Q):
    return element_diagonal(host_tangent(tmp_path, header, name, ctx, nelem, nq, passive, ai, ao, out_sizes), P, Q)


def test_a_non_symmetric_model_against_its_probed_matrix_and_host_tangent(G, tmp_path):
    from ceedpetscsolid_b200.ceed import BASIS_COLLOCATED, EVAL_GRAD, EVAL_NONE, VECTOR_ACTIVE
    (tmp_path / "nonsym.h").write_text(NONSYM)
    p, Q = 2, 3
    g = G.GpuProblem("linElas", (2, 2, 1), p, resource="/gpu/b200:jit", multigrid="none")
    d = g.fine
    K = np.random.default_rng(11).uniform(-1, 1, 81)
    K += 4 * np.eye(9).reshape(-1)
    assert rel_err(K.reshape(9, 9), K.reshape(9, 9).T) > 0.1
    ctx = (C.c_double * 81)(*K)
    qf = g.ceed.QFunction(1, f"{tmp_path / 'nonsym.h'}:NonSymdF")
    qf.add_input("du", 9, EVAL_GRAD)
    qf.add_input("qdata", 10, EVAL_NONE)
    qf.add_output("dv", 9, EVAL_GRAD)
    qf.set_context(ctx)
    op = g.ceed.Operator(qf)
    op.set_field("du", d.Erestrictu, d.basisu, VECTOR_ACTIVE)
    op.set_field("qdata", d.Erestrictqdi, BASIS_COLLOCATED, d.qdata)
    op.set_field("dv", d.Erestrictu, d.basisu, VECTOR_ACTIVE)
    assert op.is_jit_fused
    n = g.mesh.lsize(p)
    got = op_diagonal(g, op, n)
    # the dense operator, probed through K12
    assert rel_err(got, probed_diagonal(g, op, n)) < TOL
    # the host tangent, contracted and summed on the host
    nelem = g.mesh.nelem
    qd = g.strided_to_plain(d.Erestrictqdi, d.qdata)
    de = host_element_diagonal(tmp_path, "nonsym.h", "NonSymdF", ctx, nelem, Q ** 3, [qd], 0, 0, [9], p + 1, Q)
    want = np.zeros(n)
    off = g.mesh.offsets(p)
    for c in range(3):
        np.add.at(want, off + c, de[:, :, c])
    assert rel_err(got, want) < TOL


# ------------------------------------------------------------------------------- 4. models with passive fields
def test_a_model_with_passive_outputs_against_its_probed_matrix(G, tmp_path):
    """ExtraF (active fields 1 and 1, passive outputs sdiag and energy): the generic path refuses its diagonal; K14
    gives the probed one and leaves the passive outputs bitwise as an apply left them"""
    path = tmp_path / "extra.h"
    path.write_text(EXTRA_FIELDS)
    p = 2
    g = G.GpuProblem("linElas", (2, 2, 1), p, resource="/gpu/b200:jit", multigrid="none")
    nelem, Q = g.mesh.nelem, p + 1
    qd = g.strided_to_plain(g.fine.Erestrictqdi, g.fine.qdata)
    scale = np.random.default_rng(3).uniform(0, 1, (nelem, 1, Q ** 3))
    n = g.mesh.lsize(p)
    generic, _ = extra_operator(g, path, False, scale, qd)
    assert not generic.is_jit_fused
    with pytest.raises(libceed.CeedError, match="QFunction ExtraF does not qualify"):
        op_diagonal(g, generic, n)
    op, out = extra_operator(g, path, True, scale, qd)
    assert op.is_jit_fused
    want = probed_diagonal(g, op, n)
    before = {name: out(name).copy() for name in ("sdiag", "energy")}
    assert all(np.isfinite(v).all() for v in before.values())
    got = op_diagonal(g, op, n)
    assert rel_err(got, want) < TOL
    for name, v in before.items():
        np.testing.assert_array_equal(out(name).view(np.uint64), v.view(np.uint64), err_msg=name)


@pytest.mark.parametrize("P,Q", [(2, 2), (3, 3), (5, 5)])
def test_edge_model_against_its_host_tangent(tmp_path, P, Q):
    """EdgeF: 8 + 8 fields of widths 1 to 64, active fields 7 and 3, a 2048-byte context; the C entry directly"""
    from ceedpetscsolid_b200.mesh import BoxMesh
    nelem = 2 * lib.b200_elems_per_block(Q) + 1
    nq = Q ** 3
    (tmp_path / "edge.h").write_text(EDGE_FIELDS)
    rng = np.random.default_rng(P * 10 + Q)
    pin = [rng.uniform(-1, 1, (nelem, w, nq)) for w in EDGE_IN[:EDGE_AI]]
    k = rng.uniform(-1, 1, EDGE_CTX)
    k[255] = 0.0                      # the active output is then linear in the active input
    ctx = (C.c_double * EDGE_CTX)(*k)
    de = host_element_diagonal(tmp_path, "edge.h", "EdgeF", ctx, nelem, nq, pin, EDGE_AI, EDGE_AO, EDGE_OUT, P, Q)
    mesh = BoxMesh(n=(nelem, 1, 1), perturb=0.0, seed=0)
    off = mesh.offsets(P - 1)
    n = mesh.lsize(P - 1)
    want = np.zeros(n)
    for c in range(3):
        np.add.at(want, off + c, de[:, :, c])
    h = libceed.jit_diag_compile(tmp_path / "edge.h", "EdgeF", EDGE_IN, EDGE_OUT, EDGE_AI, EDGE_AO, P, Q)
    d_in = [torch.from_numpy(qblocked(a)).cuda() for a in pin]
    ptrs = [t.data_ptr() for t in d_in] + [0]
    d_off = torch.from_numpy(np.ascontiguousarray(off, dtype=np.int32)).cuda()
    got = torch.zeros(n, dtype=torch.float64, device="cuda")
    B, D = (np.ascontiguousarray(m) for m in oracle.basis_1d(P, Q, 0)[:2])
    b2(lib.b200_jit_diag_apply(h, C.addressof(ctx), C.sizeof(ctx), nelem, B.ctypes.data, D.ctypes.data,
                               d_off.data_ptr(), 8, (C.c_void_p * 8)(*ptrs), got.data_ptr(), None))
    torch.cuda.synchronize()
    assert close(got.cpu().numpy(), want), np.abs(got.cpu().numpy() - want).max()


# ------------------------------------------------------------------------------- 5. P = 2 and deterministic mode
def test_trilinear_level_is_the_diagonal_of_the_k13_matrix(pair):
    j, _ = pair("hyperFS", (3, 2, 2), 2)
    v, rows, cols = coo(j)
    A = dense(v, rows, cols, j.mesh.lsize(1))
    assert rel_err(j.diagonal(0), np.diag(A)) < TOL


def test_deterministic_diagonal_is_bit_identical_and_close_to_atomics(pair):
    jd, b = pair("hyperFS", (5, 3, 2), 4, resource="/gpu/b200:deterministic:jit")
    ja, _ = pair("hyperFS", (5, 3, 2), 4)
    assert jd.ceed.is_deterministic
    for level in range(len(jd.degrees)):
        d1, d2 = jd.diagonal(level), jd.diagonal(level)
        np.testing.assert_array_equal(d1.view(np.uint64), d2.view(np.uint64))
        assert close(d1, ja.diagonal(level))
        assert rel_err(d1, b.diagonal(level)) < TOL


# -------------------------------------------------------------------------------------------------- 6. solves
TUBE = (2, 16, 12)


def _solve(locs, coarse):
    from ceedpetscsolid_b200.elasticity import AppCtx, Elasticity
    app = AppCtx(problem="hyperFS", degree=2, num_steps=2, mesh=tube_mesh(*TUBE),
                 clamp={1: [0, 0, 0, 0, 0, 1, 0], 2: [0, -0.02, 0.04, 0, 0, 1, 0]})
    el = Elasticity(app, qf_locators=locs, coarse=coarse)
    return el, el.solve()


@pytest.mark.parametrize("coarse", ["pcg", "amg"])
def test_port_model_solves_a_tube_like_the_builtin(G, coarse):
    jel, jout = _solve(port_locators("hyperFS"), coarse)
    assert all(lv.op.is_jit_fused for lv in jel.users)
    bel, bout = _solve(None, coarse)
    assert jout["converged"] and bout["converged"]
    assert (jout["snes_its"], jout["ksp_its"]) == (bout["snes_its"], bout["ksp_its"])
    assert rel_err(jel.U.cpu().numpy(), bel.U.cpu().numpy()) < 1e-9


@pytest.mark.parametrize("coarse", ["pcg", "amg"])
def test_a_model_the_backend_does_not_have_solves_the_tube(G, tmp_path, coarse):
    h = tmp_path / "svk.h"
    h.write_text(SVK_HEADER)
    el, out = _solve({"apply": f"{h}:SvkF", "jacob": f"{h}:SvkdF"}, coarse)
    assert all(lv.op.is_jit_fused for lv in el.users)
    assert out["converged"] and out["snes_its"] >= 2
