"""Which path each operator of /gpu/b200 runs on, and what the fused operator paths check and launch: the
classification of built-in, transfer and JIT operators; the exact error messages of the element-range and partitioned
applies; the kernel launches of every operation on a built-in and a JIT Jacobian in both scatter modes; and the length
check of the diagonal, whose kernels add at the restriction's offsets."""
import functools

import numpy as np
import pytest
import torch

from ceedpetscsolid_b200 import ceed as libceed
from ceedpetscsolid_b200 import setuplibceed
from ceedpetscsolid_b200.ceed import BASIS_COLLOCATED, EVAL_GRAD, EVAL_NONE, VECTOR_ACTIVE, lib
from jit_models import EXTRA_FIELDS
from test_gpu_jit_fused import extra_operator, port_locators

pytestmark = pytest.mark.gpu
RANGE, PART = "CeedOperatorApplyAddRangeB200", "CeedOperatorApplyPartitionedB200"
DET_RANGE = ("deterministic mode: element-range applies are not supported (the ordered sum runs over the whole "
             "restriction)")


@pytest.fixture
def make(monkeypatch):
    """GpuProblem with the built-in QFunctions, or with the port models compiled through "/gpu/b200:jit"; its residual
    applied once, so the Jacobians' state (qdata, gradu) is set"""
    assert torch.cuda.is_available()
    import gpu_helpers as G

    def build(problem, n, p, jit=False, det=False, **kw):
        resource = "/gpu/b200" + (":jit" if jit else "") + (":deterministic" if det else "")
        locators = port_locators(problem) if jit else None
        with monkeypatch.context() as m:
            m.setattr(setuplibceed, "setup_all", functools.partial(setuplibceed.setup_all, qf_locators=locators))
            g = G.GpuProblem(problem, n, p, resource=resource, **kw)
        g.names = {k: v.rsplit(":", 1)[1] for k, v in setuplibceed.problem_options(problem, locators).items()
                   if k in ("apply", "jacob")}
        g.residual()
        return g
    return build


def port_jacobian(g, qdata_length):
    """the linElas port Jacobian on g's fine level, its qdata on a passive vector of qdata_length entries"""
    d = g.fine
    qf = g.ceed.QFunction(1, port_locators("linElas")["jacob"])
    qf.add_input("deltadu", 9, EVAL_GRAD)
    qf.add_input("qdata", 10, EVAL_NONE)
    qf.add_output("deltadv", 9, EVAL_GRAD)
    qf.set_context(g.phys)
    qd = g.ceed.Vector(qdata_length)
    qd.set_value(0.0)
    op = g.ceed.Operator(qf)
    op.set_field("deltadu", d.Erestrictu, d.basisu, VECTOR_ACTIVE)
    op.set_field("qdata", d.Erestrictqdi, BASIS_COLLOCATED, qd)
    op.set_field("deltadv", d.Erestrictu, d.basisu, VECTOR_ACTIVE)
    return op


def vectors(g, *lengths):
    vs = [g.ceed.Vector(n) for n in lengths]
    for v in vs:
        v.set_value(1.0)
    return vs


def raises(msg, f, *args):
    with pytest.raises(libceed.CeedError) as e:
        f(*args)
    head, _, text = str(e.value).partition("(): ")     # "libceed_b200 error 1: <file>:<line> in <function>(): "
    assert head.startswith("libceed_b200 error 1: ") and text == msg


# ------------------------------------------------------------------------------------------------ classification
@pytest.mark.parametrize("problem", ["linElas", "hyperSS", "hyperFS"])
@pytest.mark.parametrize("jit", [False, True])
def test_residual_jacobian_and_transfer_operators_classify(make, problem, jit):
    """(P, Q) = (3, 3) and (2, 3); the transfer operators keep the built-in gallery:Identity under ":jit" too"""
    g = make(problem, 2, 2, jit=jit)
    assert g.degrees == [1, 2]
    for op in (g.fine.opApply, g.data[0].opJacob, g.data[1].opJacob):
        assert (op.is_fused, op.is_jit_fused) == (not jit, jit)
    for op in (g.data[1].opProlong, g.data[1].opRestrict):
        assert (op.is_fused, op.is_jit_fused) == (True, False)


def test_jit_active_fields_away_from_field_0_and_a_short_passive_vector(make, tmp_path):
    (tmp_path / "extra.h").write_text(EXTRA_FIELDS)
    g = make("linElas", 2, 2, jit=True, multigrid="none")
    nelem, Q = g.mesh.nelem, 3
    qd_plain = g.strided_to_plain(g.fine.Erestrictqdi, g.fine.qdata)
    scale = np.random.default_rng(0).uniform(0.0, 1.0, (nelem, 1, Q ** 3))
    for blocked in (True, False):
        op, _ = extra_operator(g, tmp_path / "extra.h", blocked, scale, qd_plain)
        assert (op.is_fused, op.is_jit_fused) == (False, blocked)
    full = nelem * 10 * Q ** 3
    assert port_jacobian(g, full).is_jit_fused
    op = port_jacobian(g, full - 1)
    assert not op.is_jit_fused and not op.is_fused


# ----------------------------------------------------------------------------------------------- error messages
@pytest.mark.parametrize("jit", [False, True])
def test_range_and_partitioned_apply_messages(make, jit):
    g = make("hyperFS", 3, 2, jit=jit)            # fine (P, Q) = (3, 3): 27 elements, EB = 16
    op, name = g.fine.opJacob, g.names["jacob"]
    nelem, EB, n = g.mesh.nelem, lib.b200_elems_per_block(3), g.mesh.lsize(2)
    assert (nelem, EB) == (27, 16)
    x, y, xs, ys = vectors(g, n, n, n - 1, n - 1)
    # an operator that does not run on the fused kernels
    other = g.data[1].opProlong if not jit else port_jacobian(g, nelem * 10 * 27 - 1)
    oname = "Identity" if not jit else "port_LinElasdF"
    nx, ny = (g.mesh.lsize(1), n) if not jit else (n, n)
    ox, oy = vectors(g, nx, ny)
    raises(f"{RANGE}: operator {oname} does not run on the fused kernels", other.apply_add_range, ox, oy, 0, 16)
    raises(f"{PART}: operator {oname} does not run on the fused kernels", other.apply_partitioned, ox, oy, 0, None,
           None)
    # bad element ranges and interface counts
    for start, stop in ((5, 27), (0, 20), (0, 28), (-16, 16), (16, 0)):
        raises(f"{RANGE}: bad element range [{start}, {stop}) (nelem 27; start, and stop unless it is nelem, must be "
               f"multiples of 16)", op.apply_add_range, x, y, start, stop)
    for nif in (3, -16, 28):
        raises(f"{PART}: n_interface {nif} must be a multiple of 16 within [0, 27]", op.apply_partitioned, x, y, nif,
               None, None)
    # active vectors shorter than the L-vector
    short = f"operator {name}: active vectors shorter than the restriction's L-vector size {n}"
    for a, b in ((xs, y), (x, ys)):
        raises(short, op.apply, a, b)
        raises(short, op.apply_add, a, b)
        raises(short, op.apply_add_range, a, b, 0, 16)
        raises(short, op.apply_add_range, a, b, 16, 27)
        raises(short, op.apply_partitioned, a, b, 16, None, None)
    op.apply_add_range(xs, ys, 16, 16)             # an empty range checks nothing else
    # deterministic mode: whole ranges only, and the length is checked first
    gd = make("hyperFS", 3, 2, jit=jit, det=True)
    opd = gd.fine.opJacob
    x, y, xs = vectors(gd, n, n, n - 1)
    for start, stop in ((0, 16), (16, 27)):
        raises(DET_RANGE, opd.apply_add_range, x, y, start, stop)
        raises(short, opd.apply_add_range, xs, y, start, stop)
    opd.apply_add_range(x, y, 0, 27)
    opd.apply_partitioned(x, y, 16, None, None)    # runs as a whole


# --------------------------------------------------------------------------------------------------- launches
# kernel launches of one call after a warm-up, on the trilinear level (P, Q) = (2, 3) of hyperFS, 27 elements
OPS = ("apply", "apply_add", "apply_add_range", "apply_partitioned", "diagonal", "assemble")
LAUNCHES = {   # (jit, deterministic): launches of each operation; the ordered sum adds one in deterministic mode
    (False, False): dict(zip(OPS, (2, 2, 2, 2, 2, 1))),
    (False, True): dict(zip(OPS, (3, 3, 3, 3, 3, 1))),
    (True, False): dict(zip(OPS, (2, 2, 2, 2, 2, 2))),
    (True, True): dict(zip(OPS, (3, 3, 3, 3, 3, 2))),
}


@pytest.mark.parametrize("det", [False, True])
@pytest.mark.parametrize("jit", [False, True])
def test_launches_of_each_operation(make, jit, det):
    g = make("hyperFS", 3, 2, jit=jit, det=det)
    op = g.data[0].opJacob
    nelem, EB, n = g.mesh.nelem, lib.b200_elems_per_block(3), g.mesh.lsize(1)
    x, y, d, v = vectors(g, n, n, n, nelem * 576)
    split = [(0, nelem)] if det else [(0, EB), (EB, nelem)]
    calls = {
        "apply": lambda: op.apply(x, y),
        "apply_add": lambda: op.apply_add(x, y),
        "apply_add_range": lambda: [op.apply_add_range(x, y, a, b) for a, b in split],
        "apply_partitioned": lambda: op.apply_partitioned(x, y, EB, None, None),
        "diagonal": lambda: op.linear_assemble_diagonal(d),
        "assemble": lambda: op.linear_assemble(v),
    }
    got = {}
    for what, f in calls.items():
        f()
        n0 = libceed.launch_count()
        f()
        got[what] = libceed.launch_count() - n0
    torch.cuda.synchronize()
    assert got == LAUNCHES[jit, det], got


# ---------------------------------------------------------------------------------------------------- diagonal
@pytest.mark.parametrize("jit", [False, True])
def test_diagonal_into_a_short_vector_is_refused(make, jit):
    g = make("hyperFS", 3, 2, jit=jit)
    n = g.mesh.lsize(2)
    d, = vectors(g, n - 1)
    raises(f"CeedOperatorLinearAssembleDiagonal: operator {g.names['jacob']}: vector shorter than the restriction's "
           f"L-vector size {n}", g.fine.opJacob.linear_assemble_diagonal, d)
