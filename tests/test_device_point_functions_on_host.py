"""The arithmetic the CUDA kernels execute, checked WITHOUT a GPU: the point functions of csrc/b200_qf.cuh are
__host__ __device__; tests/c/qf_host_check.cu instantiates them for the host and this test compares them with the
reference's QFunctions (golden vectors generated from /root/reference, and the live oracle/_ref build when present):
residual F (+ stored gradu), Jacobian dF THROUGH the Jacobian cache (jcache_point + jacobian_point, the restructured
algebra and the folded quadrature weight), strain energy and the nodal diagnostics."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import make_golden  # noqa: E402
from oracle import oracle  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = np.load(os.path.join(ROOT, "tests", "golden", "qf_golden.npz"))
PROBS = {"LinElas": 0, "HyperSS": 1, "HyperFS": 2}
dp = C.POINTER(C.c_double)


@pytest.fixture(scope="module")
def hostlib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("qfhost") / "libqf_host_check.so")
    cmd = ["nvcc", "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-shared",
           "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "ceedpetscsolid_b200", "csrc"),
           os.path.join(ROOT, "tests", "c", "qf_host_check.cu"), "-o", so]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = C.CDLL(so)
    lib.qf_host_post.argtypes = [C.c_int, C.c_double, C.c_double, C.c_int, dp, dp, dp, dp]
    lib.qf_host_resjac.argtypes = [C.c_int, C.c_double, C.c_double, C.c_int, dp, dp, dp, dp, dp, dp]
    lib.qf_host_diagblocks.argtypes = [C.c_int, C.c_double, C.c_double, C.c_int, dp, dp, dp, dp]
    return lib


def _p(a):
    return a.ctypes.data_as(dp)


def _rel(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


@pytest.mark.parametrize("tag", ["katF", "rnd"])
@pytest.mark.parametrize("name", list(PROBS))
def test_residual_and_cached_jacobian_match_the_reference_qfunctions(hostlib, tag, name):
    qd = np.ascontiguousarray(GOLD[f"{tag}_qdata"])
    Q = qd.shape[1]
    du = np.ascontiguousarray(GOLD[f"{tag}_ug"].reshape(9, Q))
    ddu = np.ascontiguousarray(GOLD[f"{tag}_dug"].reshape(9, Q))
    dv, gradu, ddv = np.zeros((9, Q)), np.zeros((9, Q)), np.zeros((9, Q))
    assert hostlib.qf_host_resjac(PROBS[name], 0.3, 1.0, Q, _p(du), _p(ddu), _p(qd), _p(dv), _p(gradu), _p(ddv)) == 0
    assert _rel(dv, GOLD[f"{tag}_{name}F"]) < 1e-13
    if name != "LinElas":
        assert _rel(gradu, GOLD[f"{tag}_{name}F_gradu"]) < 1e-13
    # the Jacobian goes through the cache (16 / 10 / 9 doubles per point, weight folded into the geometry)
    assert _rel(ddv, GOLD[f"{tag}_{name}dF"]) < 5e-13, name


@pytest.mark.parametrize("scale", [1e-3, 1e-6, 1e-9])
@pytest.mark.parametrize("name", ["HyperSS", "HyperFS"])
def test_residual_keeps_relative_accuracy_at_small_strains(hostlib, name, scale):
    """The reference avoids cancellation at small strains (log1p series, det C - 1 polynomial: hyperFS.h:45-80); the
    spatial-form residual of the kernels (tau = mu (b - I) + lambda lnJ I) must do the same: relative error vs the
    reference QFunction stays at round-off however small the displacement gradient is."""
    which = oracle.default_which()
    Q, J, w, ug, _ = make_golden.rnd_inputs(Q=64, seed=5)
    phys = oracle.Physics(0.3, 1.0)
    (qd,) = oracle.call_qf("SetupGeo", which, None, Q, [J.reshape(9, Q), w.reshape(1, Q)], [10])
    du = np.ascontiguousarray(scale * ug.reshape(9, Q))
    dv_ref, gu_ref = oracle.call_qf(name + "F", which, phys, Q, [du, qd], [9, 9])
    dv, gradu, ddv = np.zeros((9, Q)), np.zeros((9, Q)), np.zeros((9, Q))
    assert hostlib.qf_host_resjac(PROBS[name], 0.3, 1.0, Q, _p(du), _p(du), _p(np.ascontiguousarray(qd)), _p(dv), _p(gradu), _p(ddv)) == 0
    assert np.abs(dv_ref).max() < 10 * scale * np.abs(qd).max() ** 2 * np.abs(ug).max()
    assert _rel(dv, dv_ref) < 5e-14, (name, scale)
    assert _rel(gradu, gu_ref) < 5e-14


@pytest.mark.parametrize("tag", ["katF", "rnd"])
@pytest.mark.parametrize("name", list(PROBS))
def test_closed_form_diagonal_blocks_equal_unit_inputs_through_the_jacobian(hostlib, tag, name):
    """k_fused_diag builds the 3x3 point blocks dW[c][d]/dH[c][d'] in closed form (diag_blocks_point); the reference's
    diagonal assembly pushes unit inputs through the Jacobian QFunction (SURVEY App. B.5).  Same numbers; also with the
    smoother's material constants (GetDiag_Ceed context swap, matops.c:215-217)."""
    qd = np.ascontiguousarray(GOLD[f"{tag}_qdata"])
    Q = qd.shape[1]
    du = np.ascontiguousarray(GOLD[f"{tag}_ug"].reshape(9, Q))
    for nu, E in ((0.3, 1.0), (0.45, 2.5)):
        closed, probed = np.zeros((27, Q)), np.zeros((27, Q))
        assert hostlib.qf_host_diagblocks(PROBS[name], nu, E, Q, _p(du), _p(qd), _p(closed), _p(probed)) == 0
        assert np.abs(probed).max() > 0
        assert _rel(closed, probed) < 1e-13, (name, nu)
        # symmetric blocks
        c = closed.reshape(3, 3, 3, Q)
        assert _rel(c, c.transpose(0, 2, 1, 3)) < 1e-13


@pytest.mark.parametrize("name", list(PROBS))
@pytest.mark.parametrize("which", ["port", "ref"])
def test_energy_and_diagnostics_match_the_reference_qfunctions(hostlib, name, which):
    if which == "ref" and not oracle.have_ref():
        # without a live build of the reference's QFunctions: their committed outputs at the committed inputs
        cases = []
        for tag in ("katF", "rnd"):
            Q = GOLD[f"{tag}_qdata"].shape[1]
            cases.append((Q, GOLD[f"{tag}_ug"].reshape(9, Q), GOLD[f"{tag}_qdata"], GOLD[f"{tag}_J"].reshape(9, Q)[3:6] - 0.1,
                          GOLD[f"{tag}_{name}Energy"], GOLD[f"{tag}_{name}Diagnostic"]))
    else:
        Q, J, w, ug, _ = make_golden.rnd_inputs(Q=48, seed=11)
        phys = oracle.Physics(0.3, 1.0)
        (qd,) = oracle.call_qf("SetupGeo", which, None, Q, [J.reshape(9, Q), w.reshape(1, Q)], [10])
        du = np.ascontiguousarray(3.0 * ug.reshape(9, Q))          # strains up to ~0.2: the series branches matter
        u = np.random.default_rng(1).standard_normal((3, Q))
        (e_ref,) = oracle.call_qf(name + "Energy", which, phys, Q, [du, qd], [1])
        (d_ref,) = oracle.call_qf(name + "Diagnostic", which, phys, Q, [u, du, qd], [8])
        cases = [(Q, du, qd, u, e_ref, d_ref)]
    for Q, du, qd, u, e_ref, d_ref in cases:
        energy, diag5 = np.zeros(Q), np.zeros((5, Q))
        assert hostlib.qf_host_post(PROBS[name], 0.3, 1.0, Q, _p(np.ascontiguousarray(du)), _p(np.ascontiguousarray(qd)),
                                    _p(energy), _p(diag5)) == 0
        assert _rel(energy, e_ref.reshape(-1)) < 1e-13
        for k in range(5):
            assert _rel(diag5[k], d_ref[3 + k]) < 1e-13, (name, k)
        assert np.array_equal(d_ref[:3], u)
