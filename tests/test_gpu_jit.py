"""User QFunctions on the device through "/gpu/b200:jit": compiled from their source file with NVRTC at operator set-up
and run by the generated point kernel (K11) on the generic operator path."""
import ctypes as C
import functools
import os
import subprocess

import numpy as np
import pytest

from helpers import PHYS, OracleProblem, rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
QF_PORT = os.path.join(ROOT, "oracle", "qf_port.c")
TOL = 1e-12
pytestmark = pytest.mark.gpu


def port_locators(problem):
    model = {"linElas": "LinElas", "hyperSS": "HyperSS", "hyperFS": "HyperFS"}[problem]
    return {"apply": f"{QF_PORT}:port_{model}F", "jacob": f"{QF_PORT}:port_{model}dF"}


@pytest.fixture
def G():
    import torch
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


# ---------------------------------------------------------------------------------------------- 1. the point kernel
POINT_HEADER = r"""#ifndef JIT_POINT_MODEL_H
#define JIT_POINT_MODEL_H
#include <ceed.h>
#include <math.h>

typedef struct PointCtx_ *PointCtx;
struct PointCtx_ {
  CeedScalar a, b, c;
  CeedInt k;
};

static inline CeedScalar sq(CeedScalar x) { return x * x; }
static inline CeedScalar dot3(const CeedScalar x[3], const CeedScalar y[3]) { return x[0] * y[0] + x[1] * y[1] + x[2] * y[2]; }

CEED_QFUNCTION(PointModel)(void *ctx, const CeedInt Q, const CeedScalar *const *in, CeedScalar *const *out) {
  const CeedScalar *w = in[0];
  const CeedScalar(*g)[3][CEED_Q_VLA] = (const CeedScalar(*)[3][CEED_Q_VLA])in[1];
  const CeedScalar(*qd)[CEED_Q_VLA] = (const CeedScalar(*)[CEED_Q_VLA])in[2];
  CeedScalar(*v)[3][CEED_Q_VLA] = (CeedScalar(*)[3][CEED_Q_VLA])out[0];
  CeedScalar(*s)[CEED_Q_VLA] = (CeedScalar(*)[CEED_Q_VLA])out[1];
  const PointCtx p = (const PointCtx)ctx;
  CeedPragmaSIMD
  for (CeedInt i = 0; i < Q; i++) {
    for (int j = 0; j < 3; j++)
      for (int l = 0; l < 3; l++) v[j][l][i] = p->a * w[i] * qd[1 + 3 * j + l][i] + p->b * qd[0][i] * g[l][j][i];
    const CeedScalar r[3] = {g[0][0][i], g[1][1][i], g[2][2][i]};
    s[0][i] = exp(p->c * dot3(r, r));
    s[1][i] = sqrt(1.0 + sq(qd[9][i]));
    s[2][i] = log1p(fabs(w[i])) * p->k;
    s[3][i] = pow(1.5 + sq(g[1][2][i]), p->c) - cos(qd[4][i]);
  }
  return 0;
}
#endif
"""


class PointCtx(C.Structure):
    _fields_ = [("a", C.c_double), ("b", C.c_double), ("c", C.c_double), ("k", C.c_int)]


def _host_point_model(tmp_path, ctx, nelem, nq, ins, out_sizes, header="point.h", name="PointModel"):
    """the same header (tmp_path / header) built with gcc against oracle/ref_shim.h (CEED_Q_VLA = Q), QFunction
    `name` run element by element"""
    shim = tmp_path / "shim"
    shim.mkdir(exist_ok=True)
    (shim / "ceed.h").write_text('#include "ref_shim.h"\n')
    drv = tmp_path / f"drv_{name}.c"
    drv.write_text(f'#include "{header}"\n'
                   f"int run(void *ctx, int Q, const double *const *in, double *const *out) {{ return {name}(ctx, Q, in, out); }}\n")
    so = tmp_path / f"lib{name}.so"
    subprocess.run(["/usr/bin/gcc", "-std=gnu99", "-O2", "-fPIC", "-shared", "-ffp-contract=off", f"-I{shim}",
                    f"-I{os.path.join(ROOT, 'oracle')}", f"-I{tmp_path}", str(drv), "-o", str(so), "-lm"], check=True)
    lib = C.CDLL(str(so))
    outs = [np.zeros((nelem, s, nq)) for s in out_sizes]
    dp = C.POINTER(C.c_double)
    for e in range(nelem):
        pin = (dp * len(ins))(*[a[e].ctypes.data_as(dp) for a in ins])
        pout = (dp * len(outs))(*[o[e].ctypes.data_as(dp) for o in outs])
        assert lib.run(C.byref(ctx), nq, pin, pout) == 0
    return outs


def test_point_kernel_equals_the_host_build_of_the_same_header(G, tmp_path):
    from ceedpetscsolid_b200 import ceed as libceed
    from ceedpetscsolid_b200.ceed import BASIS_COLLOCATED, EVAL_NONE
    (tmp_path / "point.h").write_text(POINT_HEADER)
    nelem, nq = 37, 27           # nelem * nq = 999: not a multiple of the 128-thread block
    sizes_in, sizes_out = [1, 9, 10], [9, 4]
    rng = np.random.default_rng(5)
    ins = [rng.uniform(-1, 1, (nelem, s, nq)) for s in sizes_in]
    ctx = PointCtx(0.7, -1.3, 0.45, 3)
    ref = _host_point_model(tmp_path, ctx, nelem, nq, ins, sizes_out)

    ceed = libceed.Ceed("/gpu/b200:jit")
    qf = ceed.QFunction(1, f"{tmp_path / 'point.h'}:PointModel")
    for i, s in enumerate(sizes_in):
        qf.add_input(f"in{i}", s, EVAL_NONE)
    for i, s in enumerate(sizes_out):
        qf.add_output(f"out{i}", s, EVAL_NONE)
    qf.set_context(ctx)
    op = ceed.Operator(qf)
    vin, rs = [], []
    for i, s in enumerate(sizes_in + sizes_out):
        r = ceed.StridedElemRestriction(nelem, nq, s, nelem * s * nq, strides=[1, nq, s * nq])  # [elem][comp][q]
        v = ceed.Vector(nelem * s * nq)
        if i < len(sizes_in):
            v.set_array(ins[i].reshape(-1).copy(), libceed.MEM_HOST, libceed.COPY_VALUES)
        rs.append(r)
        vin.append(v)
    for i in range(len(sizes_in)):
        op.set_field(f"in{i}", rs[i], BASIS_COLLOCATED, vin[i])
    op.set_field("out0", rs[3], BASIS_COLLOCATED, libceed.VECTOR_ACTIVE)
    op.set_field("out1", rs[4], BASIS_COLLOCATED, vin[4])
    assert not op.is_fused
    dummy = ceed.Vector(1)
    dummy.set_value(0.0)
    op.apply(dummy, vin[3])
    got = [vin[3].to_numpy().reshape(nelem, 9, nq), vin[4].to_numpy().reshape(nelem, 4, nq)]
    for k in range(2):
        assert np.max(np.abs(got[k] - ref[k])) <= 1e-13 * np.max(np.abs(ref[k])), k


# ------------------------------------------------------------------------------ 2. the stock models through the JIT
@pytest.mark.parametrize("problem,n,p", [("linElas", 3, 2), ("hyperSS", 3, 3), ("hyperFS", 2, 4)])
def test_stock_models_through_the_jit_equal_builtin_and_oracle(G, jit_problem, problem, n, p):
    g = jit_problem(problem, n, p, port_locators(problem))
    b = G.GpuProblem(problem, n, p)
    o = OracleProblem(problem, n, p)
    fine = len(g.degrees) - 1
    assert not g.fine.opApply.is_fused and not any(d.opJacob.is_fused for d in g.data)
    yo = o.residual_fine(o.u_fine)
    yg, yb = g.residual(), b.residual()
    assert rel_err(yg, yo) < TOL and rel_err(yg, yb) < TOL
    if o.has_gradu:
        gu = g.strided_to_plain(g.fine.ErestrictGradui, g.fine.gradu)
        assert rel_err(gu, o.gradu) < TOL
        assert rel_err(gu, b.strided_to_plain(b.fine.ErestrictGradui, b.fine.gradu)) < TOL
    rng = np.random.default_rng(1)
    for level, deg in enumerate(g.degrees):
        ol = OracleProblem(problem, n, p, pl=deg)
        x = rng.standard_normal(ol.lsize)
        jg = g.jacobian(level, x)
        assert rel_err(jg, ol.jacobian(x)) < TOL, level
        assert rel_err(jg, b.jacobian(level, x)) < TOL, level
        dg = g.diagonal(level)
        assert rel_err(dg, ol.diagonal()) < TOL, level
        assert rel_err(dg, b.diagonal(level)) < TOL, level
    assert fine == len(g.degrees) - 1


def test_one_compilation_per_distinct_qfunction(jit_problem, tmp_path):
    from ceedpetscsolid_b200 import ceed as libceed
    src = tmp_path / "qf_port_copy.c"     # a path of its own: a program this process has not compiled yet
    src.write_text(open(QF_PORT).read())
    n0 = libceed.jit_compile_count()
    g = jit_problem("hyperFS", 2, 4, {"apply": f"{src}:port_HyperFSF", "jacob": f"{src}:port_HyperFSdF"})
    assert g.degrees == [1, 2, 4]
    assert not g.fine.opApply.is_fused
    for d in g.data:
        assert not d.opJacob.is_fused
    assert libceed.jit_compile_count() - n0 == 2   # F once, dF once for the three p-multigrid levels


# ------------------------------------------------------------------------------------------------- 3. determinism
def test_deterministic_jit_jacobian_is_bit_identical(jit_problem):
    g = jit_problem("hyperFS", 3, 2, port_locators("hyperFS"), resource="/gpu/b200:jit:deterministic")
    assert g.ceed.is_deterministic
    g.residual()
    x = np.random.default_rng(2).standard_normal(g.mesh.lsize(2))
    fine = len(g.degrees) - 1
    y1, y2 = g.jacobian(fine, x), g.jacobian(fine, x)
    assert np.array_equal(y1, y2)
    d1, d2 = g.diagonal(fine), g.diagonal(fine)
    assert np.array_equal(d1, d2)


# ------------------------------------------------------------------------------------------------- 4. the guard case
def _patched_ceed(monkeypatch, mapping):
    """libceed.Ceed.QFunction that hands the backend a host pointer, as the reference's C code does
    (as in test_qfunction_guard.py)"""
    from ceedpetscsolid_b200 import ceed as libceed
    from oracle import oracle
    orig = libceed.Ceed.QFunction
    which = oracle.default_which()

    def with_pointer(self, vlength, source, f=None):
        name = source.split(":")[-1]
        name = mapping.get(name, name)
        ptr = oracle.qf(name, which) if name in oracle.QF_NAMES else None
        return orig(self, vlength, source, ptr)
    monkeypatch.setattr(libceed.Ceed, "QFunction", with_pointer)


def _small_strain_under_the_finite_strain_name(tmp_path):
    h = tmp_path / "hyperFS_edited.h"
    h.write_text(f'#include <ceed.h>\n#include "{QF_PORT}"\n'
                 "CEED_QFUNCTION(HyperFSdF)(void *ctx, const CeedInt Q, const CeedScalar *const *in, CeedScalar *const *out) {\n"
                 "  return port_HyperSSdF(ctx, Q, in, out);\n}\n")
    return {"jacob": f"{h}:HyperFSdF"}


def test_guard_mismatch_is_an_error_by_default(G, jit_problem, monkeypatch, tmp_path):
    from ceedpetscsolid_b200 import ceed as libceed
    _patched_ceed(monkeypatch, {"HyperFSdF": "HyperSSdF"})
    with pytest.raises(libceed.CeedError, match="does not compute what this backend's device body"):
        g = jit_problem("hyperFS", 2, 2, _small_strain_under_the_finite_strain_name(tmp_path), resource="/gpu/b200")
        g.residual()
        g.jacobian(len(g.degrees) - 1, np.zeros(g.mesh.lsize(2)))


@pytest.mark.parametrize("E", [1.0, 2.0])
def test_guard_mismatch_runs_the_source_under_jit(G, jit_problem, monkeypatch, tmp_path, E):
    """with E = 2 also: the Jacobian context is declared with the reference's 8 bytes (sizeof a pointer), and the
    guard-routed QFunction still reads E, the second double"""
    from ceedpetscsolid_b200 import setuplibceed
    from oracle import oracle
    _patched_ceed(monkeypatch, {"HyperFSdF": "HyperSSdF"})
    locs = _small_strain_under_the_finite_strain_name(tmp_path)
    with monkeypatch.context() as m:
        # the Jacobian keeps the built-in name, so set_context keeps the reference's size = 8
        m.setattr(setuplibceed, "problem_options", lambda problem, q=None: dict(setuplibceed.PROBLEM_OPTIONS[problem], **locs))
        g = G.GpuProblem("hyperFS", 2, 2, resource="/gpu/b200:jit", E=E)
    fine = len(g.degrees) - 1
    assert g.fine.opApply.is_fused and not g.data[fine].opJacob.is_fused
    g.residual()
    o = OracleProblem("hyperSS", 2, 2)   # hyperSS and hyperFS residuals store the same gradu
    x = np.random.default_rng(3).standard_normal(o.lsize)
    want = oracle.operator_apply("hyperSS", True, (PHYS[0], E), o.nelem, o.P, o.Q, o.B, o.D, o.offsets, o.qdata,
                                 o.gradu, x, o.which)
    assert rel_err(g.jacobian(fine, x), want) < TOL


# ------------------------------------------------------------------------------------------------------ 5. context
def test_context_is_reread_at_every_apply(jit_problem):
    from oracle import oracle
    g = jit_problem("hyperFS", 2, 2, port_locators("hyperFS"))
    o = OracleProblem("hyperFS", 2, 2)
    g.residual()
    fine = len(g.degrees) - 1
    x = np.random.default_rng(4).standard_normal(o.lsize)
    assert rel_err(g.jacobian(fine, x), o.jacobian(x)) < TOL
    g.phys.nu, g.phys.E = 0.25, 3.0
    want = oracle.operator_apply("hyperFS", True, (0.25, 3.0), o.nelem, o.P, o.Q, o.B, o.D, o.offsets, o.qdata,
                                 o.gradu, x, o.which)
    assert rel_err(g.jacobian(fine, x), want) < TOL
    assert rel_err(g.jacobian(fine, x), o.jacobian(x)) > 1e-3


def test_a_context_above_2kb_is_an_error(jit_problem):
    from ceedpetscsolid_b200 import ceed as libceed
    g = jit_problem("hyperFS", 2, 2, port_locators("hyperFS"))
    big = (C.c_double * 257)(0.3, 1.0)   # 2056 bytes
    g.data[-1].qfJacob.set_context(big)
    g.residual()
    with pytest.raises(libceed.CeedError, match="context of 2056 bytes; a JIT-compiled QFunction takes at most 2048"):
        g.jacobian(len(g.degrees) - 1, np.zeros(g.mesh.lsize(2)))


# -------------------------------------------------------------------------------------------------------- 6. solves
def _solve(qf_locators, assemble):
    from ceedpetscsolid_b200.elasticity import AppCtx, Elasticity
    app = AppCtx(problem="hyperFS", degree=2, n=(4, 4, 4), num_steps=2, perturb=0.05)
    el = Elasticity(app, qf_locators=qf_locators, assemble=assemble)
    out = el.solve()
    return el, out


def test_solve_with_the_port_model_matches_the_builtin_path(G):
    jel, jout = _solve(port_locators("hyperFS"), "coo")
    assert "jit" in jel.ceed.resource and jel.levels[0].coo is None   # p = 1 level not fused: assembled by colouring
    bel, bout = _solve(None, "colour")
    assert jout["converged"] and bout["converged"]
    assert (jout["snes_its"], jout["ksp_its"]) == (bout["snes_its"], bout["ksp_its"])
    assert rel_err(jel.U.cpu().numpy(), bel.U.cpu().numpy()) < 1e-9


SVK_HEADER = r"""#include <ceed.h>
#include <math.h>
/* St. Venant-Kirchhoff: S = lambda tr(E) I + 2 mu E, E = (F^T F - I) / 2, P = F S */
typedef struct { CeedScalar nu, E; } SvkPhysics;

static inline void svk_lame(const SvkPhysics *p, CeedScalar *mu, CeedScalar *lambda) {
  *mu = p->E / (2 * (1 + p->nu));
  *lambda = p->E * p->nu / ((1 + p->nu) * (1 - 2 * p->nu));
}
static inline void svk_geo(const CeedScalar (*qd)[CEED_Q_VLA], CeedInt i, CeedScalar *wdetJ, CeedScalar X[3][3]) {
  *wdetJ = qd[0][i];
  for (int a = 0; a < 3; a++)
    for (int b = 0; b < 3; b++) X[a][b] = qd[1 + 3 * a + b][i];
}
/* H[c][k] = sum_m dXdx[m][k] du[m][c] */
static inline void svk_grad(const CeedScalar (*du)[3][CEED_Q_VLA], CeedInt i, const CeedScalar X[3][3], CeedScalar H[3][3]) {
  for (int c = 0; c < 3; c++)
    for (int k = 0; k < 3; k++) {
      CeedScalar s = 0;
      for (int m = 0; m < 3; m++) s += X[m][k] * du[m][c][i];
      H[c][k] = s;
    }
}
static inline void svk_push(const CeedScalar P[3][3], const CeedScalar X[3][3], CeedScalar wdetJ, CeedInt i,
                            CeedScalar (*dv)[3][CEED_Q_VLA]) {
  for (int k = 0; k < 3; k++)
    for (int c = 0; c < 3; c++) {
      CeedScalar s = 0;
      for (int m = 0; m < 3; m++) s += X[k][m] * P[c][m];
      dv[k][c][i] = s * wdetJ;
    }
}
static inline void svk_stress(CeedScalar mu, CeedScalar lambda, const CeedScalar E[3][3], CeedScalar S[3][3]) {
  const CeedScalar tr = E[0][0] + E[1][1] + E[2][2];
  for (int a = 0; a < 3; a++)
    for (int b = 0; b < 3; b++) S[a][b] = (a == b ? lambda * tr : 0) + 2 * mu * E[a][b];
}

CEED_QFUNCTION(SvkF)(void *ctx, const CeedInt Q, const CeedScalar *const *in, CeedScalar *const *out) {
  const CeedScalar(*du)[3][CEED_Q_VLA] = (const CeedScalar(*)[3][CEED_Q_VLA])in[0];
  const CeedScalar(*qd)[CEED_Q_VLA] = (const CeedScalar(*)[CEED_Q_VLA])in[1];
  CeedScalar(*dv)[3][CEED_Q_VLA] = (CeedScalar(*)[3][CEED_Q_VLA])out[0];
  CeedScalar(*gradu)[3][CEED_Q_VLA] = (CeedScalar(*)[3][CEED_Q_VLA])out[1];
  CeedScalar mu, lambda;
  svk_lame((const SvkPhysics *)ctx, &mu, &lambda);
  CeedPragmaSIMD
  for (CeedInt i = 0; i < Q; i++) {
    CeedScalar wdetJ, X[3][3], H[3][3], F[3][3], E[3][3], S[3][3], P[3][3];
    svk_geo(qd, i, &wdetJ, X);
    svk_grad(du, i, X, H);
    for (int a = 0; a < 3; a++)
      for (int b = 0; b < 3; b++) { gradu[a][b][i] = H[a][b]; F[a][b] = H[a][b] + (a == b); }
    for (int a = 0; a < 3; a++)
      for (int b = 0; b < 3; b++) {
        CeedScalar s = 0;
        for (int m = 0; m < 3; m++) s += F[m][a] * F[m][b];
        E[a][b] = (s - (a == b)) / 2;
      }
    svk_stress(mu, lambda, E, S);
    for (int a = 0; a < 3; a++)
      for (int b = 0; b < 3; b++) {
        CeedScalar s = 0;
        for (int m = 0; m < 3; m++) s += F[a][m] * S[m][b];
        P[a][b] = s;
      }
    svk_push(P, X, wdetJ, i, dv);
  }
  return 0;
}

CEED_QFUNCTION(SvkdF)(void *ctx, const CeedInt Q, const CeedScalar *const *in, CeedScalar *const *out) {
  const CeedScalar(*ddu)[3][CEED_Q_VLA] = (const CeedScalar(*)[3][CEED_Q_VLA])in[0];
  const CeedScalar(*qd)[CEED_Q_VLA] = (const CeedScalar(*)[CEED_Q_VLA])in[1];
  const CeedScalar(*gradu)[3][CEED_Q_VLA] = (const CeedScalar(*)[3][CEED_Q_VLA])in[2];
  CeedScalar(*ddv)[3][CEED_Q_VLA] = (CeedScalar(*)[3][CEED_Q_VLA])out[0];
  CeedScalar mu, lambda;
  svk_lame((const SvkPhysics *)ctx, &mu, &lambda);
  CeedPragmaSIMD
  for (CeedInt i = 0; i < Q; i++) {
    CeedScalar wdetJ, X[3][3], dH[3][3], F[3][3], E[3][3], dE[3][3], S[3][3], dS[3][3], dP[3][3];
    svk_geo(qd, i, &wdetJ, X);
    svk_grad(ddu, i, X, dH);
    for (int a = 0; a < 3; a++)
      for (int b = 0; b < 3; b++) F[a][b] = gradu[a][b][i] + (a == b);
    for (int a = 0; a < 3; a++)
      for (int b = 0; b < 3; b++) {
        CeedScalar s = 0, ds = 0;
        for (int m = 0; m < 3; m++) { s += F[m][a] * F[m][b]; ds += dH[m][a] * F[m][b] + F[m][a] * dH[m][b]; }
        E[a][b] = (s - (a == b)) / 2;
        dE[a][b] = ds / 2;
      }
    svk_stress(mu, lambda, E, S);
    svk_stress(mu, lambda, dE, dS);
    for (int a = 0; a < 3; a++)
      for (int b = 0; b < 3; b++) {
        CeedScalar s = 0;
        for (int m = 0; m < 3; m++) s += dH[a][m] * S[m][b] + F[a][m] * dS[m][b];
        dP[a][b] = s;
      }
    svk_push(dP, X, wdetJ, i, ddv);
  }
  return 0;
}
"""


def test_a_model_the_backend_does_not_have_newton_and_central_differences(G, jit_problem, tmp_path):
    from ceedpetscsolid_b200.elasticity import AppCtx, Elasticity
    h = tmp_path / "svk.h"
    h.write_text(SVK_HEADER)
    locs = {"apply": f"{h}:SvkF", "jacob": f"{h}:SvkdF"}
    # the tangent against central differences of the residual operator, at a non-trivial state
    g = jit_problem("hyperFS", 3, 2, locs)
    fine = len(g.degrees) - 1
    u = g.u_fine * 5
    g.residual(u)
    d = np.random.default_rng(6).standard_normal(u.size) * np.abs(u).max()
    Jd = g.jacobian(fine, d)
    eps = 1e-5
    fd = (g.residual(u + eps * d) - g.residual(u - eps * d)) / (2 * eps)
    assert rel_err(Jd, fd) < 1e-6
    # Newton on a small box, two load steps
    app = AppCtx(problem="hyperFS", degree=2, n=(3, 3, 3), num_steps=2, perturb=0.05)
    out = Elasticity(app, qf_locators=locs).solve()
    assert out["converged"] and out["snes_its"] >= 2
