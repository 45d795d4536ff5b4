"""K12, the fused operator kernel generated around a JIT-compiled user QFunction (csrc/b200_jit_fused.cuh,
generated_fused in csrc/b200_jit.cu), and K11, the JIT point kernel, called through the C ABI and compared with
float64 references, with the method of tests/test_gpu_operator_kernels.py:
  * the six QFunctions of oracle/qf_port.c with the stock field shapes at every (P, Q) of B200_FOR_PQ and element
    counts 1, EB - 1, EB, EB + 1, 3 EB + 2, against the oracle running the gcc build of the same functions;
  * both scatters (FP64 atomics; the E-vector, d_y bitwise unchanged, summed with b200_transpose_gather_add);
  * element ranges advanced as include/b200_kernels.h prescribes, against the whole apply;
  * a model with 8 inputs and 8 outputs of widths 1 to 64 (tests/jit_models.py EdgeF) and a 2048-byte context,
    against the gcc build of the same header with the oracle's restriction and basis around it;
  * stored outputs prefilled with NaN, added-to outputs with known values, GUARD trailing entries that must survive;
    elementwise max |got - ref| <= 1e-12 max |ref|.
And, through the libCEED layer, CeedOperatorApplyAddRangeB200's refusal of a range that ends inside an element
group."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

from ceedpetscsolid_b200 import ceed
from ceedpetscsolid_b200.ceed import b2, lib
from ceedpetscsolid_b200.exodus import tube_mesh
from helpers import reoriented
from jit_models import EDGE_AI, EDGE_AO, EDGE_CTX, EDGE_FIELDS, EDGE_IN, EDGE_OUT
from oracle import oracle
from test_gpu_jit import _host_point_model
from test_gpu_operator_kernels import COUNTS, PAIRS, Case, addend, check, eb, rng_for, strip, to_qb
from test_gpu_primitives import GUARD_VAL, assert_bits, dev, fetch, out
from test_jit_fused_compile import QF_PORT, STOCK

pytestmark = pytest.mark.gpu

_vp, _i, _sz = ceed._vp, ceed._i, ceed._sz
ceed._proto("b200_jit_fused_apply", _i, _vp, _sz, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _vp, _i)
ceed._proto("b200_jit_apply", _i, _vp, _sz, _i, _i, _i, _vp, _i, _vp)
ceed._proto("b200_launch_count_reset", restype=None)
ceed._proto("b200_launch_count", restype=C.c_ulonglong)

PROBLEM = {"LinElas": "linElas", "HyperSS": "hyperSS", "HyperFS": "hyperFS"}


def stock_name(problem, jacobian):
    model = {v: k for k, v in PROBLEM.items()}[problem]
    return f"port_{model}{'dF' if jacobian else 'F'}"


class PortCase(Case):
    """Case whose oracle runs the gcc build of oracle/qf_port.c, the functions K12, K13 and K14 are compiled
    around"""

    def oracle_apply(self, jacobian, x, off=None):
        return oracle.operator_apply(self.problem, jacobian, self.phys, self.nelem, self.P, self.Q, self.B, self.D,
                                     self.off if off is None else off, self.qdata, self.gradu, x, which="port")

    def oracle_diagonal(self):
        return oracle.operator_diagonal(self.problem, self.phys, self.nelem, self.P, self.Q, self.B, self.D, self.off,
                                        self.qdata, self.gradu, self.lsize, which="port")


def k12(h, ctx, nelem, c, d_off, d_x, d_y, d_ev, ins, outs, padd):
    """one b200_jit_fused_apply; ins / outs: device addresses of the fields (None for the active ones)"""
    return lib.b200_jit_fused_apply(h, C.addressof(ctx), C.sizeof(ctx), nelem, c.B.ctypes.data, c.D.ctypes.data, d_off,
                                    d_x, d_y, d_ev, len(ins), (C.c_void_p * 8)(*ins), len(outs),
                                    (C.c_void_p * 8)(*outs), padd)


def ranged(c, h, ctx, ranges, d_x, ins, outs, padd):
    """launch(d_y, d_evec) for Case.scatter: K12 once per element range [e0, e1), with d_offsets, the passive fields
    ((tensor or None, width) pairs, q-blocked) and d_evec advanced to element e0"""
    P3, Q3 = c.P ** 3, c.Q ** 3

    def at(fields, e0):
        return [None if t is None else t.data_ptr() + 8 * e0 * w * Q3 for t, w in fields]

    def launch(d_y, d_ev):
        for e0, e1 in ranges:
            rc = k12(h, ctx, e1 - e0, c, c.d_off.data_ptr() + 4 * e0 * P3, d_x.data_ptr(), d_y,
                     None if d_ev is None else d_ev + 8 * e0 * 3 * P3, at(ins, e0), at(outs, e0), padd)
            if rc:
                return rc
        return 0
    return launch


def stock_fields(c, jacobian, d_gu_out):
    ins_w, outs_w = STOCK[stock_name(c.problem, jacobian)]
    d_in = [None, c.d_qd] + ([dev(to_qb(c.gradu), np.nan)] if len(ins_w) == 3 else [])
    d_out = [None] + ([d_gu_out] if len(outs_w) == 2 else [])
    return list(zip(d_in, ins_w)), list(zip(d_out, outs_w))


def run_stock(c, jacobian, scatters=(False, True), ranges=None):
    """K12 around port_*F (residual: y and the stored gradu) or port_*dF (Jacobian at the oracle's gradu) on Case c,
    one call per element range, against the oracle; returns {d_evec?: (y, gradu or None)}.  x and the addend of y
    depend on the case only, so runs over different ranges can be compared bit for bit."""
    name = stock_name(c.problem, jacobian)
    h = ceed.jit_fused_compile(QF_PORT, name, *STOCK[name], 0, 0, c.P, c.Q)
    ranges = ranges or [(0, c.nelem)]
    ngu = c.nelem * 9 * c.Q ** 3
    if jacobian:
        x = rng_for(name, c.nelem, "x").standard_normal(c.lsize)
        ref = c.oracle_apply(True, x)
    else:
        x, ref = c.u, c.r
    d_x = dev(x, np.nan)
    res = {}
    for evec in scatters:
        tag = (f"{name} at (P, Q) = ({c.P}, {c.Q}), {c.nelem} elements, ranges {ranges}, "
               f"{'d_evec' if evec else 'atomic'}")
        gu = out(ngu) if c.has_gradu and not jacobian else None
        ins, outs = stock_fields(c, jacobian, gu)
        y0 = addend(rng_for(name, c.nelem, evec), ref, c.lsize)
        y = c.scatter(ranged(c, h, c.cphys, ranges, d_x, ins, outs, 0), y0, evec)
        check(y, y0 + ref, ref, tag)
        g = None
        if gu is not None:
            g = fetch(gu, ngu)
            check(g, to_qb(c.gradu), c.gradu, f"gradu, q-blocked: {tag}")
        res[evec] = (y, g)
    return res


# --------------------------------------------------------------------------- 1. stock programs, every instantiation


@pytest.mark.parametrize("count", list(COUNTS))
@pytest.mark.parametrize("P,Q", PAIRS)
@pytest.mark.parametrize("name", sorted(STOCK))
def test_stock_programs_match_the_oracle(name, P, Q, count):
    jacobian = name.endswith("dF")
    model = name[5:-2] if jacobian else name[5:-1]
    run_stock(PortCase(PROBLEM[model], P, Q, COUNTS[count](eb(Q)), perm=count in ("EB", "3EB+2")), jacobian)


# --------------------------------------------------------------------------- 2. meshes and bases


@pytest.mark.parametrize("P,Q", [(4, 5), (3, 5)])
def test_stock_hyperfs_on_a_reoriented_tube(P, Q):
    """neighbouring elements with different local axes; 30 elements: a tail group of 2"""
    mesh = reoriented(tube_mesh(2, 5, 3), seed=4)
    c = PortCase("hyperFS", P, Q, mesh.nelem, perm=True, mesh=mesh)
    run_stock(c, False)
    run_stock(c, True)


@pytest.mark.parametrize("P,Q", [(3, 4), (4, 4)])
def test_stock_hyperfs_follows_the_basis_values(P, Q):
    """K12 derives the collocated derivative from the matrices of each call: Gauss, Gauss-Lobatto and Gauss again at
    one (P, Q), one compiled program, must each match their own oracle"""
    for qmode in (0, 1, 0):
        c = PortCase("hyperFS", P, Q, eb(Q) + 3, qmode=qmode)
        run_stock(c, False, scatters=(False,))
        run_stock(c, True, scatters=(False,))


def test_stock_hyperfs_near_incompressible():
    c = PortCase("hyperFS", 4, 5, 2 * eb(5) + 1, perm=True, nu=0.49)
    run_stock(c, False)
    run_stock(c, True)


# --------------------------------------------------------------------------- 3. element ranges at the C ABI


@pytest.mark.parametrize("jacobian", [False, True], ids=["residual", "jacobian"])
@pytest.mark.parametrize("P,Q", [(2, 3), (4, 5), (5, 5)])
@pytest.mark.parametrize("k", [1, 2])
def test_ranges_add_up_to_the_whole_apply(k, P, Q, jacobian):
    """[0, k EB) and [k EB, 3 EB + 2): the second call ends with the true tail group.  With the E-vector the two calls
    write disjoint slices of one E-vector, summed once: bit for bit the whole apply; gradu likewise"""
    EB = eb(Q)
    c = PortCase("hyperFS", P, Q, 3 * EB + 2, perm=True)
    whole = run_stock(c, jacobian)
    split = run_stock(c, jacobian, ranges=[(0, k * EB), (k * EB, c.nelem)])
    assert_bits(split[True][0], whole[True][0], "y, E-vector scatter, split vs whole")
    check(split[False][0], whole[False][0], whole[False][0], "y, atomic scatter, split vs whole")
    for evec in (False, True):
        if not jacobian:
            assert_bits(split[evec][1], whole[evec][1], "gradu, split vs whole")


# --------------------------------------------------------------------------- 4./5. field-shape edges, context


@pytest.fixture(scope="module")
def edge_dir(tmp_path_factory):
    d = tmp_path_factory.mktemp("edge")
    (d / "edge.h").write_text(EDGE_FIELDS)
    return d


def host_edge(d, ctx, nelem, nq, ins):
    """EdgeF built with gcc (test_gpu_jit._host_point_model) in a directory of its own: one library per call"""
    sub = d / f"host{len(list(d.glob('host*')))}"
    sub.mkdir()
    (sub / "edge.h").write_text(EDGE_FIELDS)
    return _host_point_model(sub, ctx, nelem, nq, ins, EDGE_OUT, header="edge.h", name="EdgeF")


class EdgeCase(Case):
    """EdgeF (tests/jit_models.py) on a strip of nelem elements with node-permuted offsets: passive inputs, the
    context, x, and the reference (E-restriction, oracle gradient, the gcc build of EdgeF, transposed gradient,
    np.add.at into the L-vector)"""

    def __init__(self, d, P, Q, nelem):
        self.d, self.P, self.Q, self.nelem = d, P, Q, nelem
        mesh = strip(nelem)
        self.rng = rng_for("edge", P, Q, nelem)
        nn = mesh.num_nodes(P - 1)
        self.lsize = 3 * nn
        self.off = mesh.offsets(P - 1, node_perm=self.rng.permutation(nn)).reshape(nelem, P ** 3)
        self.d_off = dev(self.off.reshape(-1))
        self.B, self.D = (np.ascontiguousarray(m) for m in oracle.basis_1d(P, Q, 0)[:2])
        self.x = self.rng.standard_normal(self.lsize)
        self.pin = [self.rng.uniform(-1, 1, (nelem, w, Q ** 3)) for w in EDGE_IN[:EDGE_AI]]
        self.ctx = (C.c_double * EDGE_CTX)(*self.rng.uniform(-1, 1, EDGE_CTX))

    def reference(self):
        nelem, P, Q = self.nelem, self.P, self.Q
        dofs = self.off[:, None, :] + np.arange(3)[None, :, None]                     # [e][c][node]
        du = oracle.basis_apply(nelem, 3, P, Q, self.B, self.D, None, 0, 2, self.x[dofs]).reshape(nelem, 9, Q ** 3)
        outs = host_edge(self.d, self.ctx, nelem, Q ** 3, self.pin + [du])
        ve = oracle.basis_apply(nelem, 3, P, Q, self.B, self.D, None, 1, 2, outs[EDGE_AO]).reshape(nelem, 3, P ** 3)
        y = np.zeros(self.lsize)
        np.add.at(y, dofs, ve)
        return y, outs

    def run(self, h, evec, padd):
        """K12 with either scatter, passive outputs over NaN (padd = 0) or over known values (padd = 1); checks y and
        every passive output"""
        Q3, tag = self.Q ** 3, f"EdgeF at (P, Q) = ({self.P}, {self.Q}), {self.nelem} elements, " \
                               f"{'d_evec' if evec else 'atomic'}, passive_add {padd}"
        ref, rout = self.reference()
        d_x = dev(self.x, np.nan)
        ins = [(dev(to_qb(a), np.nan), w) for a, w in zip(self.pin, EDGE_IN)] + [(None, 9)]
        outs, known = [], []
        for i, w in enumerate(EDGE_OUT):
            n = self.nelem * w * Q3
            k0 = addend(self.rng, rout[i], n).reshape(self.nelem, w, Q3) if padd else np.zeros((self.nelem, w, Q3))
            known.append(k0)
            outs.append((None if i == EDGE_AO else dev(to_qb(k0), GUARD_VAL) if padd else out(n), w))
        y0 = addend(self.rng, ref, self.lsize)
        y = self.scatter(ranged(self, h, self.ctx, [(0, self.nelem)], d_x, ins, outs, padd), y0, evec)
        check(y, y0 + ref, ref, tag)
        for i, (t, w) in enumerate(outs):
            if t is not None:
                check(fetch(t, self.nelem * w * Q3), to_qb(known[i] + rout[i]), rout[i], f"passive output {i}: {tag}")
        return y - y0


def edge_fused(d, P, Q):
    return ceed.jit_fused_compile(d / "edge.h", "EdgeF", EDGE_IN, EDGE_OUT, EDGE_AI, EDGE_AO, P, Q)


@pytest.mark.parametrize("count", ["EB-1", "2EB+1"])
@pytest.mark.parametrize("P,Q", [(2, 2), (2, 3), (5, 5)])
def test_eight_fields_of_widths_1_to_64(edge_dir, P, Q, count):
    """(2, 2): EB = 16, 64 threads; (2, 3): EB = 16, 160 threads; (5, 5): EB = 4"""
    nelem = eb(Q) - 1 if count == "EB-1" else 2 * eb(Q) + 1
    c = EdgeCase(edge_dir, P, Q, nelem)
    h = edge_fused(edge_dir, P, Q)
    for evec in (False, True):
        for padd in (0, 1):
            c.run(h, evec, padd)


def test_the_last_bytes_of_a_2kb_context_are_read_at_every_call(edge_dir):
    P, Q = 3, 4
    c = EdgeCase(edge_dir, P, Q, eb(Q) + 1)
    h = edge_fused(edge_dir, P, Q)
    y1 = c.run(h, False, 0)
    c.ctx[EDGE_CTX - 1] += 0.75
    y2 = c.run(h, False, 0)
    assert np.abs(y1 - y2).max() > 1e-3 * np.abs(y1).max()


def test_a_context_of_2049_bytes_is_refused(edge_dir):
    big = (C.c_char * 2049)()
    c = EdgeCase(edge_dir, 2, 2, 3)
    hf = edge_fused(edge_dir, 2, 2)
    hp = ceed.jit_compile(edge_dir / "edge.h", "EdgeF", EDGE_IN, EDGE_OUT)
    d_y = out(c.lsize, 0.0)
    nul = (C.c_void_p * 8)()
    for fn, call in (("b200_jit_fused_apply",
                      lambda: lib.b200_jit_fused_apply(hf, C.addressof(big), 2049, c.nelem, c.B.ctypes.data,
                                                       c.D.ctypes.data, c.d_off.data_ptr(), d_y.data_ptr(),
                                                       d_y.data_ptr(), None, 8, nul, 8, nul, 0)),
                     ("b200_jit_apply", lambda: lib.b200_jit_apply(hp, C.addressof(big), 2049, 3, 8, 8, nul, 8, nul))):
        lib.b200_launch_count_reset()
        assert call() != 0, fn
        assert f"{fn}: context of 2049 bytes; a JIT QFunction takes at most 2048" in lib.b200_last_error().decode()
        assert lib.b200_launch_count() == 0
    assert_bits(fetch(d_y, c.lsize), np.zeros(c.lsize), "y after refused calls")


# --------------------------------------------------------------------------- 6. K11


def run_k11(d, Q, nelem):
    nq = Q ** 3
    rng = rng_for("k11", Q, nelem)
    ins = [rng.uniform(-1, 1, (nelem, w, nq)) for w in EDGE_IN]
    ctx = (C.c_double * EDGE_CTX)(*rng.uniform(-1, 1, EDGE_CTX))
    ref = host_edge(d, ctx, nelem, nq, ins)
    h = ceed.jit_compile(d / "edge.h", "EdgeF", EDGE_IN, EDGE_OUT)
    d_in = [dev(a.reshape(-1), np.nan) for a in ins]
    d_out = [out(nelem * w * nq) for w in EDGE_OUT]
    b2(lib.b200_jit_apply(h, C.addressof(ctx), C.sizeof(ctx), nelem, nq, 8, (C.c_void_p * 8)(*[t.data_ptr() for t in d_in]),
                          8, (C.c_void_p * 8)(*[t.data_ptr() for t in d_out])))
    for i, (t, w) in enumerate(zip(d_out, EDGE_OUT)):
        check(fetch(t, nelem * w * nq).reshape(nelem, w, nq), ref[i], ref[i], f"K11 output {i}, Q = {Q}")


@pytest.mark.parametrize("Q", range(2, 9))
def test_k11_eight_fields_of_widths_1_to_64(edge_dir, Q):
    run_k11(edge_dir, Q, 7)


def test_k11_grid_stride_second_pass(edge_dir):
    """1190 elements of 512 points: more threads of work than the capped grid of 148 * 32 blocks of 128"""
    assert 1190 * 512 > 148 * 32 * 128
    run_k11(edge_dir, 8, 1190)


# --------------------------------------------------------------------------- 7. ranges through the libCEED layer


def ceed_vec(g, t):
    v = g.ceed.Vector(t.numel())
    v.set_array(t)
    return v


@pytest.fixture
def problem(monkeypatch):
    """GpuProblem on the 27-element box, K12 (resource "/gpu/b200:jit" with the qf_port.c locators) or built-in"""
    import gpu_helpers
    from ceedpetscsolid_b200 import setuplibceed

    def make(p, k12):
        if not k12:
            return gpu_helpers.GpuProblem("hyperFS", 3, p, multigrid="none")
        locs = {"apply": f"{QF_PORT}:port_HyperFSF", "jacob": f"{QF_PORT}:port_HyperFSdF"}
        with monkeypatch.context() as m:
            m.setattr(setuplibceed, "setup_all", functools.partial(setuplibceed.setup_all, qf_locators=locs))
            return gpu_helpers.GpuProblem("hyperFS", 3, p, multigrid="none", resource="/gpu/b200:jit")
    return make


@pytest.mark.parametrize("kind", ["residual", "jacobian", "k12_jacobian"])
@pytest.mark.parametrize("p", [4, 2], ids=["Q5_EB4", "Q3_EB16"])
def test_apply_add_range_refuses_a_stop_inside_an_element_group(problem, p, kind):
    """a range ending inside a group would run that group with the range's extent over per-point data laid out with
    the whole mesh's: refused, with the output and gradu untouched; ranges on group bounds add up to the full apply"""
    g = problem(p, kind == "k12_jacobian")
    nelem, EB = g.mesh.nelem, eb(p + 1)
    assert nelem == 27
    op = g.fine.opApply if kind == "residual" else g.fine.opJacob
    assert op.is_jit_fused == (kind == "k12_jacobian")
    g.residual()
    lsize = g.mesh.lsize(p)
    x = torch.from_numpy(g.u_fine if kind == "residual" else rng_for(kind, p).standard_normal(lsize)).cuda()
    yf = torch.zeros_like(x)
    torch.cuda.synchronize()
    xc, yc = ceed_vec(g, x), ceed_vec(g, yf)
    op.apply(xc, yc)
    yc.take_array()
    gu_full = g.fine.gradu.to_numpy()
    y0 = torch.from_numpy(addend(rng_for(kind, p, "y0"), yf.cpu().numpy(), lsize)).cuda()
    yr = y0.clone()
    torch.cuda.synchronize()
    yc.set_array(yr)
    with pytest.raises(ceed.CeedError, match=r"bad element range \[0, 13\)"):
        op.apply_add_range(xc, yc, 0, 13)
    torch.cuda.synchronize()
    assert_bits(yr.cpu().numpy(), y0.cpu().numpy(), "output after the refused call")
    assert_bits(g.fine.gradu.to_numpy(), gu_full, "gradu after the refused call")
    if kind == "residual":
        g.fine.gradu.set_value(float("nan"))
    bounds = [0, 4, 12, nelem] if EB == 4 else [0, 16, nelem]
    yr.zero_()
    torch.cuda.synchronize()
    for e0, e1 in zip(bounds[:-1], bounds[1:]):
        op.apply_add_range(xc, yc, e0, e1)
    xc.take_array()
    yc.take_array()
    torch.cuda.synchronize()
    got, want = yr.cpu().numpy(), yf.cpu().numpy()
    assert np.abs(got - want).max() <= 1e-14 * np.abs(want).max(), f"ranges {bounds} vs the full apply"
    assert_bits(g.fine.gradu.to_numpy(), gu_full, "gradu after the ranges vs after the full apply")
