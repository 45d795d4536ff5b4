"""The operator kernels of include/b200_kernels.h -- fused residual (and the gradu it stores), Jacobian cache,
Jacobian, diagonal, p-multigrid transfer, P = 2 element-matrix assembly and the generic restriction / basis
kernels -- called one by one through the C ABI and compared with the float64 oracle at the same (P, Q), offsets,
quadrature data and state.

Method (that of tests/test_gpu_primitives.py):
  * every (P, Q) of B200_FOR_PQ and every transfer pair of XF in csrc/b200_fused.cu, all three problems;
  * element counts 1, EB - 1, EB, EB + 1, 3 EB + 2 (EB = b200_elems_per_block(Q)): empty, partial and full element
    groups, with and without the tail-group launch, and one mesh of more than OFFSETS_AHEAD = 1024 groups;
  * both scatters: FP64 atomics into the L-vector, and the deterministic E-vector (d_y must stay bitwise unchanged)
    summed with b200_transpose_gather_add;
  * outputs the kernel stores to are prefilled with NaN, outputs it adds to with known values, and every output
    carries GUARD trailing entries that must survive;
  * elementwise max |got - ref| <= 1e-12 max |ref| per output (ref without the prefilled addend), so one wrong
    entry fails."""
import ctypes as C
import zlib

import numpy as np
import pytest
import torch

from ceedpetscsolid_b200 import ceed
from ceedpetscsolid_b200.ceed import b2, lib
from ceedpetscsolid_b200.exodus import tube_mesh
from ceedpetscsolid_b200.mesh import BoxMesh
from helpers import reoriented
from oracle import oracle
from test_gpu_primitives import GUARD_VAL, assert_bits, dev, fetch, map_build, out

pytestmark = pytest.mark.gpu

# entry points that the package itself does not call through ctypes
_vp, _i, _ll = ceed._vp, ceed._i, ceed._ll
ceed._proto("b200_apply_residual", _i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp)
ceed._proto("b200_apply_jacobian", _i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp)
ceed._proto("b200_apply_diagonal", _i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp)
ceed._proto("b200_jcache_build", _i, _i, _i, _vp, _vp, _vp)
ceed._proto("b200_assemble_p1", _i, _vp, _i, _i, _vp, _vp, _vp, _vp)
ceed._proto("b200_restrict_strided", _i, _i, _i, _i, _i, _ll, _ll, _ll, _vp, _vp)
ceed._proto("b200_basis_apply", _i, _i, _i, _i, _vp, _vp, _vp, _i, _i, _vp, _vp)
ceed._proto("b200_transpose_gather_add", _i, _vp, _vp, _i, _i, _i, _i, _vp, _vp)

PROBLEMS = ["linElas", "hyperSS", "hyperFS"]
PID = {"linElas": 0, "hyperSS": 1, "hyperFS": 2}
PAIRS = [(2, 2), (2, 3), (3, 3), (2, 4), (3, 4), (4, 4), (2, 5), (3, 5), (4, 5), (5, 5)]   # B200_FOR_PQ
XF = [(2, 3), (3, 4), (4, 5), (3, 5), (2, 4), (2, 5)]                                      # b200_apply_transfer
COUNTS = {"1": lambda eb: 1, "EB-1": lambda eb: eb - 1, "EB": lambda eb: eb, "EB+1": lambda eb: eb + 1,
          "3EB+2": lambda eb: 3 * eb + 2}
OFFSETS_AHEAD = 1024
TOL = 1e-12


def rng_for(*key):
    return np.random.default_rng(zlib.crc32(repr(key).encode()))


def eb(Q):
    return lib.b200_elems_per_block(Q)


def qblocked_index(nelem, ncomp, Q):
    """[elem][comp][q] -> position in the q-blocked backend layout (mirror of qblocked_index, csrc/b200_common.cuh;
    the scalar mirror is tests/test_abi_and_layout.py::_qblocked)"""
    EB, T, Q3 = eb(Q), Q * Q, Q ** 3
    e = np.arange(nelem, dtype=np.int64)[:, None, None]
    c = np.arange(ncomp, dtype=np.int64)[None, :, None]
    q = np.arange(Q3, dtype=np.int64)[None, None, :]
    g, ei = e // EB, e % EB
    ebn = np.minimum(EB, nelem - g * EB)
    return g * EB * ncomp * Q3 + (c * Q + q % Q) * (ebn * T) + (q // Q) * ebn + ei


def to_qb(a):
    nelem, ncomp, Q3 = a.shape
    v = np.full(a.size, np.nan)
    v[qblocked_index(nelem, ncomp, round(Q3 ** (1 / 3)))] = a
    return v


def check(got, ref, scale, what):
    """max |got - ref| <= TOL max|scale| elementwise; NaN fails"""
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    lim = TOL * np.abs(scale).max()
    err = np.abs(got - ref)
    bad = np.flatnonzero(~(err <= lim))
    assert bad.size == 0, (f"{what}: {bad.size} of {got.size} entries off; first at {bad[0]}: {got.flat[bad[0]]!r} vs "
                           f"{ref.flat[bad[0]]!r}, worst {np.nanmax(err):.3g} (bound {lim:.3g})")


def addend(rng, scale, n):
    """known non-zero values for the outputs a kernel adds to"""
    return np.abs(scale).max() * rng.integers(-4, 5, n) / 4.0


def strip(nelem, h=0.5):
    """a row of nelem perturbed cubes of side h: exact element counts.  Every vertex of a strip lies on its boundary,
    which BoxMesh(perturb=...) leaves in place, so the vertices are moved here: with cubes, every element would have
    the same diagonal dX/dx, and a kernel that swapped x and y nodes, or elements, could still match"""
    box = BoxMesh(n=(nelem, 1, 1), lengths=(h * nelem, h, h))
    V = box.vertices + 0.1 * h * (rng_for("strip", nelem).random(box.vertices.shape) - 0.5)
    return BoxMesh(n=(nelem, 1, 1), lengths=(h * nelem, h, h), vertices=V)


def ptr(t):
    return None if t is None else t.data_ptr()


class Case:
    """state of one (problem, P, Q, mesh) on the host: oracle residual (which writes gradu), quadrature data"""

    def __init__(self, problem, P, Q, nelem, perm=False, nu=0.3, qmode=0, mesh=None):
        self.problem, self.pid, self.P, self.Q, self.nelem = problem, PID[problem], P, Q, nelem
        self.mesh = mesh if mesh is not None else strip(nelem)
        self.rng = rng_for(problem, P, Q, nelem, perm, nu, qmode)
        nn = self.mesh.num_nodes(P - 1)
        self.lsize = 3 * nn
        self.off = self.mesh.offsets(P - 1, node_perm=self.rng.permutation(nn) if perm else None)
        self.B, self.D = (np.ascontiguousarray(m) for m in oracle.basis_1d(P, Q, qmode)[:2])
        self.qdata = oracle.setup_geo(nelem, Q, self.mesh.offsets(1), self.mesh.coord_lvector())
        self.has_gradu = oracle.PROBLEMS[problem][2]
        self.gradu = np.zeros((nelem, 9, Q ** 3)) if self.has_gradu else None
        self.phys = (nu, 1.0)
        self.cphys = ceed.Physics(nu, 1.0)
        self.u = 2e-4 * self.rng.standard_normal(self.lsize)        # small displacement: det F stays near 1
        self.r = self.oracle_apply(False, self.u)
        self.d_off = dev(self.off.reshape(-1))
        self.d_qd = dev(to_qb(self.qdata), np.nan)

    def oracle_apply(self, jacobian, x, off=None):
        return oracle.operator_apply(self.problem, jacobian, self.phys, self.nelem, self.P, self.Q, self.B, self.D,
                                     self.off if off is None else off, self.qdata, self.gradu, x)

    def oracle_diagonal(self):
        return oracle.operator_diagonal(self.problem, self.phys, self.nelem, self.P, self.Q, self.B, self.D, self.off,
                                        self.qdata, self.gradu, self.lsize)

    def head(self):
        return (self.pid, C.addressof(self.cphys), self.nelem, self.P, self.Q, self.B.ctypes.data, self.D.ctypes.data,
                self.d_off.data_ptr())

    def scatter(self, launch, y0, evec):
        """run launch(d_y, d_evec) with either scatter; returns the L-vector"""
        n = self.lsize
        d_y = dev(y0, GUARD_VAL)
        if not evec:
            b2(launch(d_y.data_ptr(), None))
            return fetch(d_y, n)
        ev = out(self.nelem * 3 * self.P ** 3)
        b2(launch(d_y.data_ptr(), ev.data_ptr()))
        assert_bits(fetch(d_y, n), y0, "d_y with d_evec given")
        fetch(ev, self.nelem * 3 * self.P ** 3)
        ordered_add(n, self.off, self.P ** 3, ev, d_y)
        return fetch(d_y, n)

    def jcache(self, gradu_dev):
        nj = lib.b200_jcache_ncomp(self.pid) * self.nelem * self.Q ** 3
        jc = out(nj)
        b2(lib.b200_jcache_build(self.pid, self.nelem, self.Q, self.d_qd.data_ptr(), ptr(gradu_dev), jc.data_ptr()))
        assert np.isfinite(fetch(jc, nj)).all(), "Jacobian cache entries left unwritten"
        return jc


def probed_element_matrices(c):
    """[e][col][row] = K_e[row, col] of a P = 2 case, element dof node*3 + comp: 24 unit probes of the case's oracle
    Jacobian on the same elements with every element's nodes its own (offsets = arange(8 nelem) * 3)"""
    own = (np.arange(c.nelem * 8, dtype=np.int32) * 3).reshape(c.nelem, 8)
    ref = np.empty((c.nelem, 24, 24))
    for col in range(24):
        x = np.zeros(c.nelem * 24)
        x[col::24] = 1.0
        ref[:, col, :] = c.oracle_apply(True, x, own).reshape(c.nelem, 24)
    return ref


def ordered_add(lsize, off, elemsize, ev, d_y):
    rc, tptr, tidx = map_build(lsize, off.reshape(-1))
    assert rc == 0
    b2(lib.b200_transpose_gather_add(lsize, dev(tptr).data_ptr(), dev(tidx, 0).data_ptr(), elemsize, 3, 1, 1,
                                     ev.data_ptr(), d_y.data_ptr()))


def run_operator_kernels(c, scatters=(False, True)):
    """residual + gradu, Jacobian cache from the kernel's and from the oracle's gradu, Jacobian, diagonal"""
    Q3 = c.Q ** 3
    d_x = dev(c.u, np.nan)
    x = c.rng.standard_normal(c.lsize)
    d_xj = dev(x, np.nan)
    jref = c.oracle_apply(True, x)
    dref = c.oracle_diagonal()
    d_gu_oracle = dev(to_qb(c.gradu), np.nan) if c.has_gradu else None
    for evec in scatters:
        tag = "d_evec" if evec else "atomic"
        y0 = addend(c.rng, c.r, c.lsize)
        d_gu = out(c.nelem * 9 * Q3) if c.has_gradu else None
        y = c.scatter(lambda dy, ev: lib.b200_apply_residual(*c.head(), c.d_qd.data_ptr(), ptr(d_gu), d_x.data_ptr(),
                                                              dy, ev), y0, evec)
        check(y, y0 + c.r, c.r, f"residual ({tag})")
        if c.has_gradu:
            check(fetch(d_gu, c.nelem * 9 * Q3), to_qb(c.gradu), c.gradu, f"gradu, q-blocked ({tag})")
        sources = [("kernel gradu", d_gu), ("oracle gradu", d_gu_oracle)] if c.has_gradu else [("", None)]
        for name, src in sources:
            jc = c.jcache(src)
            y0 = addend(c.rng, jref, c.lsize)
            y = c.scatter(lambda dy, ev: lib.b200_apply_jacobian(*c.head(), jc.data_ptr(), d_xj.data_ptr(), dy, ev),
                          y0, evec)
            check(y, y0 + jref, jref, f"Jacobian, cache from {name} ({tag})")
        y0 = addend(c.rng, dref, c.lsize)
        y = c.scatter(lambda dy, ev: lib.b200_apply_diagonal(*c.head(), jc.data_ptr(), dy, ev), y0, evec)
        check(y, y0 + dref, dref, f"diagonal ({tag})")


# --------------------------------------------------------------------------- a. fused operator kernels


@pytest.mark.parametrize("count", list(COUNTS))
@pytest.mark.parametrize("P,Q", PAIRS)
@pytest.mark.parametrize("problem", PROBLEMS)
def test_fused_operator_kernels_match_the_oracle(problem, P, Q, count):
    run_operator_kernels(Case(problem, P, Q, COUNTS[count](eb(Q)), perm=count in ("EB", "3EB+2")))


@pytest.mark.parametrize("problem,P,Q", [("linElas", 3, 4), ("hyperSS", 2, 3), ("hyperFS", 4, 5)])
def test_fused_operator_kernels_near_incompressible(problem, P, Q):
    run_operator_kernels(Case(problem, P, Q, 2 * eb(Q) + 1, perm=True, nu=0.49))


def test_fused_operator_kernels_past_the_offsets_prefetch_distance():
    """more than OFFSETS_AHEAD full groups: the CTAs that prefetch the offsets of a later group run"""
    Q = 3
    run_operator_kernels(Case("hyperFS", 2, Q, (OFFSETS_AHEAD + 6) * eb(Q) + 5, perm=True))


# --------------------------------------------------------------------------- b. basis cache


@pytest.mark.parametrize("P,Q", [(3, 4), (4, 4)])
def test_basis_cache_follows_the_basis_values(P, Q):
    """cached_mats<P, Q> is keyed on the interp / grad values: Gauss, Gauss-Lobatto, Gauss again at one (P, Q)
    must each match their own oracle (a stale collocated derivative would not)"""
    nelem = eb(Q) + 3
    for qmode in (0, 1, 0):
        run_operator_kernels(Case("hyperFS", P, Q, nelem, qmode=qmode), scatters=(False,))


# --------------------------------------------------------------------------- c. transfer


def transfer_case(Pc, Pf, nelem, perm):
    mesh = strip(nelem)
    rng = rng_for(Pc, Pf, nelem, perm)
    nf = mesh.num_nodes(Pf - 1)
    offc = mesh.offsets(Pc - 1)
    offf = mesh.offsets(Pf - 1, node_perm=rng.permutation(nf) if perm else None)
    lc, lf = mesh.lsize(Pc - 1), 3 * nf
    J = np.ascontiguousarray(oracle.basis_1d(Pc, Pf, 1)[0])
    minv = 1.0 / oracle.multiplicity(nelem, Pf ** 3, 3, lf, offf)
    return rng, offc, offf, lc, lf, J, minv


TRANSFER_MODES = [(d, m) for d in ("prolong", "restrict") for m in ("plain", "mult", "inject") if
                  not (d == "restrict" and m == "inject")]


@pytest.mark.parametrize("direction,mode", TRANSFER_MODES)
@pytest.mark.parametrize("Pc,Pf", XF)
def test_transfer_matches_the_oracle(Pc, Pf, direction, mode):
    nelem = 2 * eb(Pf) + 3
    rng, offc, offf, lc, lf, J, minv = transfer_case(Pc, Pf, nelem, perm=mode == "mult")
    tr = direction == "restrict"
    nin, nout = (lf, lc) if tr else (lc, lf)
    off_out, elemsize_out = (offc, Pc ** 3) if tr else (offf, Pf ** 3)
    xin = rng.standard_normal(nin)
    d_in, d_offc, d_offf = dev(xin, np.nan), dev(offc.reshape(-1)), dev(offf.reshape(-1))
    d_mult = dev(minv, np.nan) if mode != "plain" else None
    if tr:
        ref = oracle.transfer(True, nelem, Pc, Pf, offc, offf, xin * minv if mode == "mult" else xin, lc)
    else:
        ref = oracle.transfer(False, nelem, Pc, Pf, offc, offf, xin, lf)
        if mode != "plain":
            ref = ref * minv
    launch = lambda d_out, ev: lib.b200_apply_transfer(int(tr), nelem, Pc, Pf, J.ctypes.data, d_offc.data_ptr(),
                                                       d_offf.data_ptr(), ptr(d_mult), int(mode == "inject"),
                                                       d_in.data_ptr(), d_out, ev)
    if mode == "inject":
        # stores, no sum: every fine node is overwritten (NaN junk before), no pre-zeroed output needed
        d_out = out(nout)
        b2(launch(d_out.data_ptr(), None))
        check(fetch(d_out, nout), ref, ref, "injected prolongation")
        return
    for evec in (False, True):
        y0 = addend(rng, ref, nout)
        d_out = dev(y0, GUARD_VAL)
        if not evec:
            b2(launch(d_out.data_ptr(), None))
        else:
            ev = out(nelem * 3 * elemsize_out)
            b2(launch(d_out.data_ptr(), ev.data_ptr()))
            assert_bits(fetch(d_out, nout), y0, "output with d_evec given")
            fetch(ev, nelem * 3 * elemsize_out)
            ordered_add(nout, off_out, elemsize_out, ev, d_out)
        check(fetch(d_out, nout), y0 + ref, ref, f"{direction} {mode} ({'d_evec' if evec else 'atomic'})")


def test_inject_is_refused_on_the_host_unless_it_is_a_scaled_prolongation():
    J = np.zeros(15)
    for transpose, mult in ((0, None), (1, 8), (1, None)):
        lib.b200_launch_count_reset()
        rc = lib.b200_apply_transfer(transpose, 5, 3, 5, J.ctypes.data, None, None, mult, 1, None, None, None)
        assert rc != 0
        assert "inject is the prolongation with multiplicity scaling" in lib.b200_last_error().decode()
        assert lib.b200_launch_count() == 0


# --------------------------------------------------------------------------- d. P = 2 element matrices


@pytest.mark.parametrize("Q", [2, 3, 4, 5])
@pytest.mark.parametrize("problem", PROBLEMS)
def test_assemble_p1_element_matrices(problem, Q):
    """d_values[(e*24 + col)*24 + row] = K_e[row, col], element dof node*3 + comp, against probed_element_matrices"""
    nelem = 2 * eb(Q) + 3
    c = Case(problem, 2, Q, nelem)
    d_gu = dev(to_qb(c.gradu), np.nan) if c.has_gradu else None
    jc = c.jcache(d_gu)
    n = nelem * 24 * 24
    vals = out(n)
    b2(lib.b200_assemble_p1(c.pid, C.addressof(c.cphys), nelem, Q, c.B.ctypes.data, c.D.ctypes.data, jc.data_ptr(),
                            vals.data_ptr()))
    ref = probed_element_matrices(c)
    check(fetch(vals, n).reshape(nelem, 24, 24), ref, ref, "element matrices")


# --------------------------------------------------------------------------- e. injected prolongation's premise


def backend_interp(P, Q, qmode):
    """interp1d of the backend's own CeedBasisCreateTensorH1Lagrange (what the transfer operators are given)"""
    c = ceed.Ceed("/gpu/b200")
    b = c.BasisTensorH1Lagrange(3, 3, P, Q, qmode)
    B = np.ascontiguousarray(b.interp1d)
    b.destroy()
    c.destroy()
    return B


def element_interpolants(Pc, Pf, mesh):
    """per-element interpolant [e][node][comp] of the NON-injected prolongation (d_mult = NULL, d_evec) with the
    backend's interpolation matrix, and the fine dof of every entry"""
    nelem = mesh.nelem
    offc, offf = mesh.offsets(Pc - 1), mesh.offsets(Pf - 1)
    J = backend_interp(Pc, Pf, ceed.GAUSS_LOBATTO)
    xc = rng_for(Pc, Pf, nelem).standard_normal(mesh.lsize(Pc - 1))
    d_in, d_offc, d_offf = dev(xc, np.nan), dev(offc.reshape(-1)), dev(offf.reshape(-1))
    d_out = dev(np.zeros(mesh.lsize(Pf - 1)), GUARD_VAL)
    n = nelem * 3 * Pf ** 3
    ev = out(n)
    b2(lib.b200_apply_transfer(0, nelem, Pc, Pf, J.ctypes.data, d_offc.data_ptr(), d_offf.data_ptr(), None, 0,
                               d_in.data_ptr(), d_out.data_ptr(), ev.data_ptr()))
    vals = fetch(ev, n)
    dof = (offf.reshape(-1, 1) + np.arange(3)).reshape(-1)
    return vals, dof


def copies_that_differ(vals, dof):
    """number of fine dofs whose element copies are not all bitwise equal"""
    order = np.argsort(dof, kind="stable")
    d, v = dof[order], vals[order].view(np.uint64)
    first = np.searchsorted(d, d, side="left")
    return np.unique(d[v != v[first]]).size, np.unique(d).size


@pytest.mark.parametrize("qmode", [ceed.GAUSS, ceed.GAUSS_LOBATTO], ids=["gauss", "lobatto"])
def test_lagrange_basis_is_a_unit_vector_at_its_own_nodes(qmode):
    """where a point coincides with a node, interp1d holds exactly that unit vector (the Lagrange recurrence alone
    gives 1 + 2^-52 at the end point of (P, Q) = (4, 5), among others); elsewhere it agrees with the oracle"""
    for P in range(2, 11):
        for Q in range(2, 11):
            B = backend_interp(P, Q, qmode)
            Bo, _, qref, _ = oracle.basis_1d(P, Q, qmode)
            nodes = oracle.lobatto(P)[0]
            for i, j in zip(*np.nonzero(qref[:, None] == nodes[None, :])):
                assert np.array_equal(B[i], np.eye(P)[j]), (P, Q, i, j, B[i])
            assert np.abs(B - Bo).max() <= 1e-14, (P, Q)


@pytest.mark.parametrize("Pc,Pf", XF)
def test_element_interpolants_agree_bitwise_on_a_box(Pc, Pf):
    """every element sharing a fine node of a box mesh (all elements in the same orientation) computes the same
    interpolant there, bit for bit: what the injected prolongation relies on"""
    vals, dof = element_interpolants(Pc, Pf, BoxMesh(n=(3, 2, 2), perturb=0.1, seed=2))
    assert copies_that_differ(vals, dof)[0] == 0


@pytest.mark.parametrize("Pc,Pf", XF)
def test_element_interpolants_on_a_reoriented_mesh(Pc, Pf):
    """neighbours with different local axes sum the same terms in another order: their copies of a shared fine dof
    differ in the last bits.  This is a property of the kernel's contraction order, recorded here; the prolongation
    therefore does not inject in deterministic mode (test_gpu_deterministic.py)"""
    vals, dof = element_interpolants(Pc, Pf, reoriented(tube_mesh(2, 6, 2), seed=5))
    ndiff, nshared = copies_that_differ(vals, dof)
    print(f"(Pc, Pf) = ({Pc}, {Pf}): {ndiff} of {nshared} fine dofs have element copies that differ")
    assert ndiff > 0
    # they differ by rounding only
    order = np.argsort(dof, kind="stable")
    d, v = dof[order], vals[order]
    first = np.searchsorted(d, d, side="left")
    assert np.abs(v - v[first]).max() <= 1e-14 * np.abs(vals).max()


# --------------------------------------------------------------------------- f. generic path


GENERIC = [(2, 3), (3, 3), (4, 3)]   # (p, qextra): (P, Q) = (3, 6), (4, 7), (5, 8)


@pytest.mark.parametrize("p,qextra", GENERIC)
@pytest.mark.parametrize("problem", PROBLEMS)
def test_generic_path_residual_jacobian_diagonal(problem, p, qextra):
    import gpu_helpers as G
    from helpers import OracleProblem
    g = G.GpuProblem(problem, 2, p, qextra=qextra, multigrid="none")
    o = OracleProblem(problem, 2, p, qextra=qextra)
    assert not g.fine.opApply.is_fused and not g.data[0].opJacob.is_fused
    r = o.residual_fine(o.u_fine)
    check(g.residual(), r, r, "residual")
    x = np.random.default_rng(p).standard_normal(o.lsize)
    j = o.jacobian(x)
    check(g.jacobian(0, x), j, j, "Jacobian")
    d = o.diagonal()
    check(g.diagonal(0), d, d, "diagonal")


@pytest.mark.parametrize("ncomp", [3, 10])
@pytest.mark.parametrize("Q", [2, 3, 4, 5, 6, 7, 8])
def test_restrict_strided_q_blocked(Q, ncomp):
    nelem = 2 * eb(Q) + 3
    Q3 = Q ** 3
    n = nelem * ncomp * Q3
    rng = rng_for(Q, ncomp, 30)
    idx = qblocked_index(nelem, ncomp, Q).reshape(-1)
    L = rng.standard_normal(n)
    E = out(n)
    b2(lib.b200_restrict_strided(0, nelem, Q3, ncomp, Q, 0, 0, 0, dev(L, np.nan).data_ptr(), E.data_ptr()))
    assert_bits(fetch(E, n), L[idx], "L -> E")
    Ein, L0 = rng.standard_normal(n), addend(rng, 1.0, n)
    d_L = dev(L0, GUARD_VAL)
    b2(lib.b200_restrict_strided(1, nelem, Q3, ncomp, Q, 0, 0, 0, dev(Ein, np.nan).data_ptr(), d_L.data_ptr()))
    ref = L0.copy()
    ref[idx] += Ein
    assert_bits(fetch(d_L, n), ref, "E -> L (adds)")


BASIS_PQ = [(2, 2), (3, 5), (5, 3), (4, 9), (10, 10), (10, 6), (6, 10)]


@pytest.mark.parametrize("P,Q", BASIS_PQ)
def test_basis_apply_matches_the_oracle(P, Q):
    nelem, ncomp = 5, 3
    B, D, _, qw = oracle.basis_1d(P, Q, 0)
    d_B, d_D, d_w = dev(B.reshape(-1)), dev(D.reshape(-1)), dev(qw)
    rng = rng_for(P, Q, 31)
    for emode, ndir in ((1, 1), (2, 3), (4, 0)):
        for tr in (0, 1):
            if emode == 4:
                u, nout = None, nelem * Q ** 3
            elif tr:
                u, nout = rng.standard_normal(nelem * ndir * ncomp * Q ** 3), nelem * ncomp * P ** 3
            else:
                u, nout = rng.standard_normal(nelem * ncomp * P ** 3), nelem * ndir * ncomp * Q ** 3
            ref = oracle.basis_apply(nelem, ncomp, P, Q, B, D, qw, tr, emode, u).reshape(-1)
            v = out(nout)
            b2(lib.b200_basis_apply(nelem, ncomp, P, Q, d_B.data_ptr(), d_D.data_ptr(), d_w.data_ptr(), tr, emode,
                                    ptr(dev(u, np.nan)) if u is not None else None, v.data_ptr()))
            check(fetch(v, nout), ref, ref, f"emode {emode} transpose {tr}")


def test_fused_dispatch_agrees_with_fused_supported():
    """b200_apply_residual accepts exactly the (P, Q) that b200_fused_supported reports; an unsupported pair is an
    error from the host and launches nothing"""
    phys = ceed.Physics(0.3, 1.0)
    dummy = dev(np.zeros(8))
    for P in range(1, 10):
        for Q in range(1, 10):
            B = np.ascontiguousarray(oracle.basis_1d(P, Q, 0)[0]) if P >= 2 else np.zeros((Q, P))
            D = np.ascontiguousarray(oracle.basis_1d(P, Q, 0)[1]) if P >= 2 else np.zeros((Q, P))
            lib.b200_launch_count_reset()
            rc = lib.b200_apply_residual(0, C.addressof(phys), 0, P, Q, B.ctypes.data, D.ctypes.data, dummy.data_ptr(),
                                         dummy.data_ptr(), None, dummy.data_ptr(), dummy.data_ptr(), None)
            supported = lib.b200_fused_supported(P, Q) == 1
            assert (rc == 0) == supported, (P, Q, lib.b200_last_error())
            assert supported == ((P, Q) in PAIRS)
            if not supported:
                assert "not instantiated" in lib.b200_last_error().decode()
            assert lib.b200_launch_count() == 0
    torch.cuda.synchronize()
