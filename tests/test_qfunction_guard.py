"""The QFunction hand-off (setuplibceed.c:370-372, 518-520, 818-820): the reference passes a host function pointer and
a "file:Name" locator; /gpu/b200 dispatches on the name to a hand-written device body.  Two safeguards:

* CPU: the generic device bodies, evaluated on the host by b200_qfunction_apply_host (the same __host__ __device__
  code the kernel runs), equal the reference's QFunctions on random points;
* GPU: at operator set-up the backend runs the CALLER'S pointer on a few known points and refuses to continue when
  it does not compute what the device body computes (a locally modified header would otherwise be ignored silently).
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import make_golden  # noqa: E402
from oracle import oracle  # noqa: E402

dp = C.POINTER(C.c_double)
QF_ID = {"SetupGeo": 1, "LinElasF": 2, "LinElasdF": 3, "HyperSSF": 4, "HyperSSdF": 5, "HyperFSF": 6, "HyperFSdF": 7}


def _host_eval(lib, name, ctx, Q, ins, out_sizes):
    ins = [np.ascontiguousarray(a, dtype=np.float64) for a in ins]
    outs = [np.zeros((s, Q)) for s in out_sizes]
    pin = (dp * len(ins))(*[a.ctypes.data_as(dp) for a in ins])
    pout = (dp * len(outs))(*[a.ctypes.data_as(dp) for a in outs])
    h = (C.c_double * 2)(*ctx) if ctx else None
    lib.b200_qfunction_apply_host.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                              C.c_int, C.c_void_p]
    rc = lib.b200_qfunction_apply_host(QF_ID[name], h, 2 if ctx else 0, 0, 1, Q, len(ins), pin, len(outs), pout)
    assert rc == 0
    return outs


def _check_device_bodies(lib, J, w, ug, dug, reference):
    """the device bodies evaluated on the host against reference(name, inputs, output sizes) -> outputs"""
    Q = w.size
    (qd,) = reference("SetupGeo", [J.reshape(9, Q), w.reshape(1, Q)], [10])
    (qd_b,) = _host_eval(lib, "SetupGeo", None, Q, [J.reshape(9, Q), w.reshape(1, Q)], [10])
    assert np.max(np.abs(qd_b - qd)) <= 1e-13 * np.max(np.abs(qd))
    du, ddu = ug.reshape(9, Q), dug.reshape(9, Q)
    for model, has_gradu in (("LinElas", False), ("HyperSS", True), ("HyperFS", True)):
        outs_ref = reference(model + "F", [du, qd], [9, 9] if has_gradu else [9])
        outs = _host_eval(lib, model + "F", (0.3, 1.0), Q, [du, qd], [9, 9] if has_gradu else [9])
        for a, b in zip(outs, outs_ref):
            assert np.max(np.abs(a - b)) <= 1e-13 * np.max(np.abs(b)), model
        jin = [ddu, qd] + ([outs_ref[1]] if has_gradu else [])
        (dv_ref,) = reference(model + "dF", jin, [9])
        (dv,) = _host_eval(lib, model + "dF", (0.3, 1.0), Q, jin, [9])
        assert np.max(np.abs(dv - dv_ref)) <= 5e-13 * np.max(np.abs(dv_ref)), model


@pytest.mark.parametrize("which", ["port", "ref"])
def test_device_bodies_evaluated_on_the_host_equal_the_reference_qfunctions(which):
    from ceedpetscsolid_b200 import ceed as libceed
    if which == "ref" and not oracle.have_ref():
        # no live build of the reference's QFunctions: their committed outputs at the committed inputs
        gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "qf_golden.npz"))
        for tag in ("katF", "rnd"):
            outs = {"SetupGeo": [gold[f"{tag}_qdata"]]}
            for model in ("LinElas", "HyperSS", "HyperFS"):
                outs[model + "F"] = [gold[f"{tag}_{model}F"]] + ([gold[f"{tag}_{model}F_gradu"]] if model != "LinElas" else [])
                outs[model + "dF"] = [gold[f"{tag}_{model}dF"]]
            J, w, ug, dug = (gold[f"{tag}_{k}"] for k in ("J", "w", "ug", "dug"))
            _check_device_bodies(libceed.lib, J, w, ug, dug, lambda name, ins, sizes: outs[name])
        return
    Q, J, w, ug, dug = make_golden.rnd_inputs(Q=40, seed=3)
    phys = oracle.Physics(0.3, 1.0)
    _check_device_bodies(libceed.lib, J, w, ug, dug,
                         lambda name, ins, sizes: oracle.call_qf(name, which, None if name == "SetupGeo" else phys, Q, ins, sizes))


def _patched_ceed(monkeypatch, mapping):
    """libceed.Ceed.QFunction that hands the backend a host pointer, as the reference's C code does"""
    from ceedpetscsolid_b200 import ceed as libceed
    orig = libceed.Ceed.QFunction
    which = oracle.default_which()

    def with_pointer(self, vlength, source, f=None):
        name = source.split(":")[-1]
        name = mapping.get(name, name)
        ptr = oracle.qf(name, which) if name in oracle.QF_NAMES else None
        return orig(self, vlength, source, ptr)
    monkeypatch.setattr(libceed.Ceed, "QFunction", with_pointer)


@pytest.mark.gpu
def test_matching_user_qfunctions_pass_the_guard(monkeypatch):
    import gpu_helpers as G
    from helpers import OracleProblem, rel_err
    _patched_ceed(monkeypatch, {})
    g = G.GpuProblem("hyperFS", 2, 2)
    o = OracleProblem("hyperFS", 2, 2)
    assert rel_err(g.residual(), o.residual_fine(o.u_fine)) < 1e-12
    x = np.random.default_rng(0).standard_normal(o.lsize)
    assert rel_err(g.jacobian(len(g.degrees) - 1, x), o.jacobian(x)) < 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("stage,mapping", [("residual", {"HyperFSF": "HyperSSF"}), ("jacobian", {"HyperFSdF": "HyperSSdF"})])
def test_a_user_qfunction_that_differs_from_the_device_body_is_refused(monkeypatch, stage, mapping):
    """a locally modified qfunctions header (here: the small-strain model under the finite-strain name)"""
    import gpu_helpers as G
    from ceedpetscsolid_b200 import ceed as libceed
    _patched_ceed(monkeypatch, mapping)
    with pytest.raises(libceed.CeedError, match="does not compute what this backend's device body"):
        g = G.GpuProblem("hyperFS", 2, 2)
        g.residual()
        g.jacobian(len(g.degrees) - 1, np.zeros(g.mesh.lsize(2)))
