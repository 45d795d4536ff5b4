"""K13, the trilinear element-matrix kernel (csrc/b200_jit_assemble.cuh), and K14, the operator-diagonal kernel
(csrc/b200_jit_diag.cuh), generated around a JIT-compiled user QFunction, called through the C ABI
(b200_jit_assemble_apply, b200_jit_diag_apply) and compared with float64 references, with the method of
tests/test_gpu_operator_kernels.py:
  * the stock Jacobians of oracle/qf_port.c (port_LinElasdF, port_HyperSSdF, port_HyperFSdF at the oracle's gradu):
    K14 at every (P, Q) of B200_FOR_PQ, K13 at (2, Q), Q = 2..5, element counts 1, EB - 1, EB, EB + 1, 3 EB + 2, against
    the oracle running the gcc build of the same functions (its diagonal for K14; for K13, 24 unit probes of its
    Jacobian on element-private offsets);
  * every extent of the tail group, EB + r elements for r = 2..EB - 1 (r = 1 is EB + 1 above): K14 at Q = 3 and 5
    (EB = 16 and 4), K13 at Q = 2 and 3, where the point tangents are walked in chunks of 128 that most extents do not
    divide;
  * K14 with both scatters: FP64 atomics onto known values, and the E-vector (d_diag bitwise unchanged) summed with
    b200_transpose_gather_add; node-permuted offsets at EB and 3 EB + 2;
  * a linear model with a non-symmetric point tangent (tests/jit_models.py NONSYM), against the gcc build of the same
    header contracted on the host: where a transposed or swapped tangent index shows;
  * the Gauss basis in every case above; Gauss-Lobatto and nu = 0.49 once per kernel;
  * the context limit: 2048 bytes accepted, 2049 refused with nothing launched and the output untouched;
  * outputs the kernels store to are prefilled with NaN, outputs they add to with known values, and every output carries
    GUARD trailing entries that must survive; elementwise max |got - ref| <= 1e-12 max |ref|.
Programs are compiled once per process for each (model, P, Q)."""
import ctypes as C

import numpy as np
import pytest

from ceedpetscsolid_b200 import ceed
from ceedpetscsolid_b200.ceed import b2, lib
from helpers import rel_err
from jit_models import NONSYM, NONSYM_CTX, NONSYM_IN, NONSYM_OUT
from test_gpu_jit_assemble import element_matrices
from test_gpu_jit_diag import element_diagonal, host_tangent
from test_gpu_jit_kernels import PortCase
from test_gpu_operator_kernels import COUNTS, PAIRS, Case, addend, check, eb, probed_element_matrices, rng_for, to_qb
from test_gpu_primitives import assert_bits, dev, fetch, out
from test_jit_fused_compile import QF_PORT, STOCK

pytestmark = pytest.mark.gpu

JACOBIANS = {"port_LinElasdF": "linElas", "port_HyperSSdF": "hyperSS", "port_HyperFSdF": "hyperFS"}
# (P, Q) and EB = b200_elems_per_block(Q) of the tail-extent cases, one Q per EB
K14_TAILS = [((3, 3), 16), ((5, 5), 4)]
K13_TAILS = [(2, 16), (3, 16)]


def pointers(fields):
    return (C.c_void_p * 8)(*[None if t is None else t.data_ptr() for t in fields])


def stock_inputs(c, name):
    """device inputs of a port_*dF: the active gradient (ignored), q-blocked qdata and, for the hyperelastic models,
    the oracle's gradu, q-blocked; each followed by NaN guards"""
    ins = [None, c.d_qd]
    if len(STOCK[name][0]) == 3:
        ins.append(dev(to_qb(c.gradu), np.nan))
    return ins


def k14(h, ctx, c, ins):
    """launch(d_diag, d_evec) for Case.scatter"""
    return lambda d_diag, d_ev: lib.b200_jit_diag_apply(h, C.addressof(ctx), C.sizeof(ctx), c.nelem, c.B.ctypes.data,
                                                        c.D.ctypes.data, c.d_off.data_ptr(), len(ins), pointers(ins),
                                                        d_diag, d_ev)


def k13_call(h, ctx, c, ins, d_values):
    return lib.b200_jit_assemble_apply(h, C.addressof(ctx), C.sizeof(ctx), c.nelem, c.B.ctypes.data, c.D.ctypes.data,
                                       len(ins), pointers(ins), d_values)


def run_k14(c, h, ctx, ins, ref, tag):
    """K14 with either scatter onto known values against ref, the L-vector diagonal"""
    for evec in (False, True):
        y0 = addend(rng_for(tag, evec), ref, c.lsize)
        y = c.scatter(k14(h, ctx, c, ins), y0, evec)
        check(y, y0 + ref, ref, f"{tag}, {'d_evec' if evec else 'atomic'}")


def run_k13(c, h, ctx, ins, ref, tag):
    """K13 into a NaN-filled output against ref [e][col][row]"""
    n = c.nelem * 576
    vals = out(n)
    b2(k13_call(h, ctx, c, ins, vals.data_ptr()))
    check(fetch(vals, n).reshape(c.nelem, 24, 24), ref, ref, tag)


def stock_k14(name, P, Q, nelem, **kw):
    c = PortCase(JACOBIANS[name], P, Q, nelem, **kw)
    h = ceed.jit_diag_compile(QF_PORT, name, *STOCK[name], 0, 0, P, Q)
    run_k14(c, h, c.cphys, stock_inputs(c, name), c.oracle_diagonal(),
            f"K14 {name} at (P, Q) = ({P}, {Q}), {nelem} elements, {kw}")


def stock_k13(name, Q, nelem, **kw):
    c = PortCase(JACOBIANS[name], 2, Q, nelem, **kw)
    h = ceed.jit_assemble_compile(QF_PORT, name, *STOCK[name], 0, 0, 2, Q)
    run_k13(c, h, c.cphys, stock_inputs(c, name), probed_element_matrices(c),
            f"K13 {name} at Q = {Q}, {nelem} elements, {kw}")


# --------------------------------------------------------------------------- 1. K14, stock Jacobians


@pytest.mark.parametrize("count", list(COUNTS))
@pytest.mark.parametrize("P,Q", PAIRS)
@pytest.mark.parametrize("name", sorted(JACOBIANS))
def test_k14_stock_jacobians_match_the_oracle(name, P, Q, count):
    stock_k14(name, P, Q, COUNTS[count](eb(Q)), perm=count in ("EB", "3EB+2"))


@pytest.mark.parametrize("P,Q,r", [(P, Q, r) for (P, Q), EB in K14_TAILS for r in range(2, EB)])
@pytest.mark.parametrize("name", sorted(JACOBIANS))
def test_k14_every_tail_group_extent(name, P, Q, r):
    """one full group and a tail group of r elements: the tail kernel's plane stride ebn T and lane t ebn + eb"""
    EB = dict(K14_TAILS)[(P, Q)]
    assert eb(Q) == EB
    stock_k14(name, P, Q, EB + r)


# --------------------------------------------------------------------------- 2. K13, stock Jacobians


@pytest.mark.parametrize("count", list(COUNTS))
@pytest.mark.parametrize("Q", [2, 3, 4, 5])
@pytest.mark.parametrize("name", sorted(JACOBIANS))
def test_k13_stock_jacobians_match_the_oracle(name, Q, count):
    stock_k13(name, Q, COUNTS[count](eb(Q)))


@pytest.mark.parametrize("Q,r", [(Q, r) for Q, EB in K13_TAILS for r in range(2, EB)])
@pytest.mark.parametrize("name", sorted(JACOBIANS))
def test_k13_every_tail_group_extent(name, Q, r):
    """one full group and a tail group of r elements: at Q = 3 the r Q^3 positions of the tail are walked in chunks of
    128, and a chunk starts on every residue mod r; at Q = 2 they fit in one chunk"""
    EB = dict(K13_TAILS)[Q]
    assert eb(Q) == EB
    stock_k13(name, Q, EB + r)


# --------------------------------------------------------------------------- 3. basis and material edges


@pytest.mark.parametrize("qmode,nu", [(ceed.GAUSS_LOBATTO, 0.3), (ceed.GAUSS, 0.49)], ids=["lobatto", "nu0.49"])
def test_k14_lobatto_basis_and_near_incompressible(qmode, nu):
    stock_k14("port_HyperFSdF", 4, 5, 2 * eb(5) + 1, perm=True, qmode=qmode, nu=nu)


@pytest.mark.parametrize("qmode,nu", [(ceed.GAUSS_LOBATTO, 0.3), (ceed.GAUSS, 0.49)], ids=["lobatto", "nu0.49"])
def test_k13_lobatto_basis_and_near_incompressible(qmode, nu):
    stock_k13("port_HyperFSdF", 3, 2 * eb(3) + 1, qmode=qmode, nu=nu)


# --------------------------------------------------------------------------- 4. a non-symmetric linear model


class NonSym:
    """NONSYM with a random non-symmetric K (the context) on 3 EB + 2 elements with node-permuted offsets; the host
    tangent at the points of each Q, built once with gcc and shared by every P"""

    def __init__(self, d):
        self.d = d
        (d / "nonsym.h").write_text(NONSYM)
        K = rng_for("nonsym").uniform(-1, 1, NONSYM_CTX) + 4 * np.eye(9).reshape(-1)
        self.ctx = (C.c_double * NONSYM_CTX)(*K)
        self.tangents = {}

    def case(self, P, Q):
        c = Case("linElas", P, Q, 3 * eb(Q) + 2, perm=True)
        if Q not in self.tangents:
            sub = self.d / f"Q{Q}"
            sub.mkdir()
            (sub / "nonsym.h").write_text(NONSYM)
            Dt = host_tangent(sub, "nonsym.h", "NonSymdF", self.ctx, c.nelem, Q ** 3, [c.qdata], 0, 0, NONSYM_OUT)
            # [e][q][s = m*3 + b][o = k*3 + a]: the whole tangent and its blocks b = a, the ones the diagonal reads
            assert rel_err(Dt, Dt.swapaxes(2, 3)) > 0.1
            Dc = np.einsum("eqmckc->eqmkc", Dt.reshape(c.nelem, Q ** 3, 3, 3, 3, 3))
            assert rel_err(Dc, Dc.swapaxes(2, 3)) > 0.1
            self.tangents[Q] = (c.qdata, Dt)
        qdata, Dt = self.tangents[Q]
        assert_bits(c.qdata, qdata, "qdata of the host tangent")
        return c, Dt

    def compile(self, kind, P, Q):
        fn = ceed.jit_diag_compile if kind == "diag" else ceed.jit_assemble_compile
        return fn(self.d / "nonsym.h", "NonSymdF", NONSYM_IN, NONSYM_OUT, 0, 0, P, Q)


@pytest.fixture(scope="module")
def nonsym(tmp_path_factory):
    return NonSym(tmp_path_factory.mktemp("nonsym"))


@pytest.mark.parametrize("P,Q", PAIRS)
def test_k14_non_symmetric_tangent(nonsym, P, Q):
    c, Dt = nonsym.case(P, Q)
    de = element_diagonal(Dt, P, Q)
    ref = np.zeros(c.lsize)
    for comp in range(3):
        np.add.at(ref, c.off + comp, de[:, :, comp])
    run_k14(c, nonsym.compile("diag", P, Q), nonsym.ctx, [None, c.d_qd], ref,
            f"K14 NonSymdF at (P, Q) = ({P}, {Q}), {c.nelem} elements")


@pytest.mark.parametrize("Q", [2, 3, 4, 5])
def test_k13_non_symmetric_tangent(nonsym, Q):
    c, Dt = nonsym.case(2, Q)
    run_k13(c, nonsym.compile("assemble", 2, Q), nonsym.ctx, [None, c.d_qd],
            element_matrices(Dt, Q).reshape(c.nelem, 24, 24), f"K13 NonSymdF at Q = {Q}, {c.nelem} elements")


# --------------------------------------------------------------------------- 5. context limit


@pytest.mark.parametrize("kernel", ["k13", "k14"])
def test_a_2048_byte_context_is_accepted_and_2049_refused(kernel):
    """the Physics constants at the front of a 2048-byte context give the oracle's result; one byte more is refused
    before anything is launched or written"""
    name, P, Q = "port_HyperFSdF", 2 if kernel == "k13" else 3, 3
    c = PortCase("hyperFS", P, Q, eb(Q) + 3, perm=True)
    ins = stock_inputs(c, name)
    ctx = (C.c_ubyte * 2048)(*rng_for("ctx").integers(0, 256, 2048).tolist())
    C.memmove(ctx, C.addressof(c.cphys), C.sizeof(c.cphys))
    big = (C.c_ubyte * 2049)()
    if kernel == "k14":
        h = ceed.jit_diag_compile(QF_PORT, name, *STOCK[name], 0, 0, P, Q)
        run_k14(c, h, ctx, ins, c.oracle_diagonal(), "K14 with a 2048-byte context")
        nev = c.nelem * 3 * P ** 3
        y0 = addend(rng_for("y0"), 1.0, c.lsize)
        d_y, d_ev = dev(y0), out(nev)
        calls = [lambda: k14(h, big, c, ins)(d_y.data_ptr(), None),
                 lambda: k14(h, big, c, ins)(d_y.data_ptr(), d_ev.data_ptr())]
        kept = [(d_y, y0), (d_ev, np.full(nev, np.nan))]
        fn = "b200_jit_diag_apply"
    else:
        h = ceed.jit_assemble_compile(QF_PORT, name, *STOCK[name], 0, 0, 2, Q)
        run_k13(c, h, ctx, ins, probed_element_matrices(c), "K13 with a 2048-byte context")
        d_v = out(c.nelem * 576)
        calls = [lambda: k13_call(h, big, c, ins, d_v.data_ptr())]
        kept = [(d_v, np.full(c.nelem * 576, np.nan))]
        fn = "b200_jit_assemble_apply"
    for call in calls:
        lib.b200_launch_count_reset()
        assert call() != 0
        assert f"{fn}: context of 2049 bytes; a JIT QFunction takes at most 2048" in lib.b200_last_error().decode()
        assert lib.b200_launch_count() == 0
    for t, want in kept:
        assert_bits(fetch(t, want.size), want, "an output after the refused calls")
