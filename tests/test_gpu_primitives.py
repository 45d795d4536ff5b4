"""The solver-side kernels of include/b200_kernels.h, called one by one through the C ABI and compared with plain
float64 references: BLAS-1 and index maps, the deterministic reductions, the device-scalar Krylov steps, the
Chebyshev smoother, the lattice transfers, the 27-point stencil and ELL mat-vecs, the ordered sums (transposed
restriction, halo unpack, level-0 AMG assembly) and the AMG block kernels.

Method:
  * exact inputs (small integers, powers of two, the lattice weights 1/2): every product and partial sum is exact, so
    the kernel must equal the reference bit for bit whatever its summation order -- a lost, doubled or misplaced term
    shows up exactly;
  * random inputs: elementwise |got - ref| <= k u sum|terms| (u = 2^-53); FMA contraction is on, so only the ordered
    pure sums are compared bitwise on random data;
  * outputs are prefilled with NaN (an entry never written fails), entries that must stay untouched hold a distinct
    value, and every output buffer carries GUARD trailing entries that must survive;
  * lengths run over SIZES, which straddle one block, the fixed reduction grid (592 x 256 threads) and the capped
    vector grid (148 * 32 blocks of 256 threads), so second and later grid-stride passes run.
Only in-range indices are passed to the device; the range checks are tested where they happen, on the host."""
import ctypes as C
import math
import zlib

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from ceedpetscsolid_b200 import ceed
from ceedpetscsolid_b200.ceed import b2, lib
from ceedpetscsolid_b200.exodus import tube_mesh
from ceedpetscsolid_b200.mesh import BoxMesh
from ceedpetscsolid_b200.solver import (ChebyshevJacobi, Vec, _guarded_ratio, _lattice_prolong_cpu,
                                        _lattice_restrict_cpu)
from helpers import dense_from_stencil, lattice_ids

pytestmark = pytest.mark.gpu

# entry points that the package itself does not call through ctypes
ceed._proto("b200_fill_strided", ceed._vp, ceed._d, ceed._sz, ceed._sz, ceed._sz)
ceed._proto("b200_transpose_gather_add", ceed._i, ceed._vp, ceed._vp, ceed._i, ceed._i, ceed._i, ceed._i, ceed._vp,
            ceed._vp)
ceed._proto("b200_transpose_map_build", ceed._i, ceed._sz, ceed._vp, ceed._vp, ceed._vp)

U = 2.0 ** -53
VEC_THREADS = 148 * 32 * 256      # capped grid of the vector kernels (256 threads per block)
RED_THREADS = 592 * 256           # fixed grid of the reductions
SIZES = [0, 1, 255, 256, 257, RED_THREADS - 1, RED_THREADS, RED_THREADS + 1, VEC_THREADS - 1, VEC_THREADS,
         VEC_THREADS + 1, 3 * VEC_THREADS + 7]
GUARD = 4
GUARD_VAL = -7.25          # tail of every output buffer
UNTOUCHED = 12345.5        # entries a kernel must leave alone (never equal to an integer test value)
# device copies made since the last fetch(): a pointer passed inline to a launch must not be handed to the next
# copy by the caching allocator before the kernel has run
_alive = []


# --------------------------------------------------------------------------- helpers


def rng_for(*key):
    return np.random.default_rng(zlib.crc32(repr(key).encode()))


def ints(rng, n, lim=2 ** 16):
    return rng.integers(-lim, lim + 1, n).astype(np.float64)


def pow2(rng, n):
    """+-2^k, |k| <= 4: products with any finite scalar of moderate size are exact"""
    return rng.choice([-1.0, 1.0], n) * 2.0 ** rng.integers(-4, 5, n)


def randn(rng, n):
    """random FP64 spanning a few decades"""
    return rng.standard_normal(n) * 10.0 ** rng.integers(-3, 4, n)


def dev(a, tail=None):
    """device copy of a host array; with `tail`, GUARD extra entries of that value follow (an input read past its
    end then poisons the result)"""
    a = np.ascontiguousarray(a)
    if tail is not None:
        a = np.concatenate([a, np.full(GUARD, tail, dtype=a.dtype)])
    t = torch.from_numpy(a).cuda()
    _alive.append(t)
    return t


def out(n, fill=np.nan):
    """device output of n entries prefilled with `fill`, followed by GUARD entries of GUARD_VAL"""
    return dev(np.full(n, fill, dtype=np.float64), tail=GUARD_VAL)


def fetch(t, n=None):
    """host copy of a device buffer after the queued work; with n, checks the guard tail and returns the body"""
    torch.cuda.synchronize()
    _alive.clear()
    h = t.cpu().numpy()
    if n is None:
        return h
    assert (h[n:] == GUARD_VAL).all(), "the kernel wrote past the end of its output"
    return h[:n]


def assert_bits(got, ref, what=""):
    got = np.ascontiguousarray(got, dtype=np.float64)
    ref = np.ascontiguousarray(ref, dtype=np.float64)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    bad = np.flatnonzero(got.view(np.uint64) != ref.view(np.uint64))
    assert bad.size == 0, (f"{what}: {bad.size} of {got.size} entries differ; first at {bad[0]}: "
                           f"{got[bad[0]]!r} != {ref[bad[0]]!r}")


def assert_within(got, ref, scale, k, what=""):
    """|got - ref| <= k u scale elementwise (scale: sum of the absolute terms of each entry); NaN fails"""
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    lim = k * U * np.asarray(scale)
    bad = np.flatnonzero(~(np.abs(got - ref) <= lim))
    assert bad.size == 0, (f"{what}: {bad.size} of {got.size} entries off; first at {bad[0]}: {got[bad[0]]!r} vs "
                           f"{ref[bad[0]]!r} (bound {np.broadcast_to(lim, got.shape)[bad[0]]:.3g})")


# --------------------------------------------------------------------------- BLAS-1 and maps, bit-exact


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("value", [0.0, -2.5], ids=["zero", "nonzero"])
def test_vec_set(n, value):
    d = out(n)
    b2(lib.b200_vec_set(d.data_ptr(), value, n))
    assert_bits(fetch(d, n), np.full(n, value))


@pytest.mark.parametrize("n", SIZES)
def test_vec_scale_and_pointwise_mult(n):
    rng = rng_for(n, 1)
    x, y = ints(rng, n), ints(rng, n)
    d = dev(x, GUARD_VAL)
    b2(lib.b200_vec_scale(d.data_ptr(), -0.75, n))
    assert_bits(fetch(d, n), x * -0.75, "scale")
    w = out(n)
    b2(lib.b200_vec_pointwise_mult(w.data_ptr(), dev(x, np.nan).data_ptr(), dev(y, np.nan).data_ptr(), n))
    assert_bits(fetch(w, n), x * y, "pointwise_mult")


RECIP_SPECIAL = np.array([0.0, -0.0, 1e-14, -1e-14, np.nextafter(1e-14, 0), np.nextafter(1e-14, 1),
                          -np.nextafter(1e-14, 0), -np.nextafter(1e-14, 1), 5e-324, -5e-324, 2.2250738585072014e-308,
                          -2.225e-308, 1e-300, np.inf, -np.inf, 1.0, -1.0, 3.0, -7.0, 0.1, 1e300, -1e-13])


@pytest.mark.parametrize("n", SIZES)
def test_vec_reciprocal_follows_the_oracle_rule(n):
    """oracle/ceed_cpu.c CeedVectorReciprocal: |v| > 1e-14 ? 1/v : v"""
    rng = rng_for(n, 2)
    x = rng.standard_normal(n) * 10.0 ** rng.integers(-16, 16, n)
    if n:
        pos = rng.choice(n, min(n, 4 * RECIP_SPECIAL.size), replace=False)
        x[pos] = np.resize(RECIP_SPECIAL, pos.size)
    d = dev(x, GUARD_VAL)
    b2(lib.b200_vec_reciprocal(d.data_ptr(), n))
    with np.errstate(divide="ignore"):
        ref = np.where(np.abs(x) > 1e-14, 1.0 / x, x)
    assert_bits(fetch(d, n), ref)


@pytest.mark.parametrize("n", SIZES)
def test_gather_scatter_maps(n):
    rng = rng_for(n, 3)
    m = n + n // 3 + 5
    src_m = ints(rng, m)
    src_n = ints(rng, n)
    idx = rng.integers(0, m, n).astype(np.int32)
    uniq = rng.permutation(m)[:n].astype(np.int32)
    holes = idx.copy()
    holes[rng.random(n) < 0.25] = -1
    d_src_m, d_src_n = dev(src_m, np.nan), dev(src_n, np.nan)
    # gather: dst[i] = src[idx[i]]
    dst = out(n)
    b2(lib.b200_gather(dst.data_ptr(), d_src_m.data_ptr(), dev(idx).data_ptr(), n))
    assert_bits(fetch(dst, n), src_m[idx], "gather")
    # scatter_set (unique indices): dst[idx[i]] = src[i], the other entries untouched
    dst = out(m, UNTOUCHED)
    b2(lib.b200_scatter_set(dst.data_ptr(), dev(uniq).data_ptr(), d_src_n.data_ptr(), n))
    ref = np.full(m, UNTOUCHED)
    ref[uniq] = src_n
    assert_bits(fetch(dst, m), ref, "scatter_set")
    # gather_or_zero: dst[i] = idx[i] >= 0 ? src[idx[i]] : 0
    dst = out(n)
    b2(lib.b200_gather_or_zero(dst.data_ptr(), d_src_m.data_ptr(), dev(holes).data_ptr(), n))
    assert_bits(fetch(dst, n), np.where(holes >= 0, src_m[np.maximum(holes, 0)], 0.0), "gather_or_zero")
    # copy_where: dst[i] = src[idx[i]] where idx[i] >= 0, untouched elsewhere
    dst = out(n, UNTOUCHED)
    b2(lib.b200_copy_where(dst.data_ptr(), d_src_m.data_ptr(), dev(holes).data_ptr(), n))
    assert_bits(fetch(dst, n), np.where(holes >= 0, src_m[np.maximum(holes, 0)], UNTOUCHED), "copy_where")
    # mask_zero: d[idx[i]] = 0, the other entries untouched
    dst = dev(src_m, GUARD_VAL)
    b2(lib.b200_mask_zero(dst.data_ptr(), dev(uniq).data_ptr(), n))
    ref = src_m.copy()
    ref[uniq] = 0.0
    assert_bits(fetch(dst, m), ref, "mask_zero")


FILL_CASES = ([(n, n + 3, 2) for n in SIZES] +
              [(1, 2, 5), (3, 7, 4), (255, 256, 17), (256, 1000, 3), (257, 258, 1), (RED_THREADS, RED_THREADS + 1, 9),
               (VEC_THREADS + 1, VEC_THREADS + 2, 3), (0, 5, 4), (2, 3, 0)])


@pytest.mark.parametrize("n,stride,count", FILL_CASES)
def test_fill_strided_leaves_the_gaps(n, stride, count):
    total = stride * count
    d = out(total, UNTOUCHED)
    b2(lib.b200_fill_strided(d.data_ptr(), -3.5, n, stride, count))
    ref = np.full(total, UNTOUCHED)
    for c in range(count):
        ref[c * stride:c * stride + n] = -3.5
    assert_bits(fetch(d, total), ref)


# --------------------------------------------------------------------------- BLAS-1, rounding bound


@pytest.mark.parametrize("n", SIZES)
def test_axpy_aypx_axpby(n):
    rng = rng_for(n, 4)
    x, y = randn(rng, n), randn(rng, n)
    a, b = -0.7, 1.3
    d_x = dev(x, np.nan)
    d_y = dev(y, GUARD_VAL)
    b2(lib.b200_vec_axpy(d_y.data_ptr(), a, d_x.data_ptr(), n))
    assert_within(fetch(d_y, n), y + a * x, np.abs(y) + np.abs(a * x), 4, "axpy")
    d_y = dev(y, GUARD_VAL)
    b2(lib.b200_vec_aypx(d_y.data_ptr(), a, d_x.data_ptr(), n))
    assert_within(fetch(d_y, n), x + a * y, np.abs(x) + np.abs(a * y), 4, "aypx")
    z = out(n)
    b2(lib.b200_vec_axpby(z.data_ptr(), a, d_x.data_ptr(), b, dev(y, np.nan).data_ptr(), n))
    assert_within(fetch(z, n), a * x + b * y, np.abs(a * x) + np.abs(b * y), 4, "axpby")


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("data", ["int", "random"])
def test_scatter_add_with_repeated_indices(n, data):
    rng = rng_for(n, 5, data)
    m = n // 5 + 1
    idx = rng.integers(0, m, n).astype(np.int32)
    gen = ints if data == "int" else randn
    dst0, src = gen(rng, m), gen(rng, n)
    d = dev(dst0, GUARD_VAL)
    b2(lib.b200_scatter_add(d.data_ptr(), dev(idx).data_ptr(), dev(src, np.nan).data_ptr(), n))
    got = fetch(d, m)
    ref = dst0.copy()
    np.add.at(ref, idx, src)
    if data == "int":
        assert_bits(got, ref)
    else:   # atomics: any order; both sums carry at most (terms) roundings
        scale = np.abs(dst0)
        np.add.at(scale, idx, np.abs(src))
        terms = np.bincount(idx, minlength=m) + 1
        assert_within(got, ref, scale, 2 * terms + 2)


# --------------------------------------------------------------------------- reductions


def dot_dev(x, y, n, w=None):
    r = dev(np.array([np.nan]))
    if w is None:
        b2(lib.b200_vec_dot(x.data_ptr(), y.data_ptr(), n, r.data_ptr()))
    else:
        b2(lib.b200_vec_dot_weighted(w.data_ptr(), x.data_ptr(), y.data_ptr(), n, r.data_ptr()))
    return fetch(r)[0]


def dot_host(x, y, n):
    r = C.c_double(np.nan)
    b2(lib.b200_vec_dot_host(x.data_ptr(), y.data_ptr(), n, C.byref(r)))
    return r.value


def norm_host(x, n, kind):
    r = C.c_double(np.nan)
    b2(lib.b200_vec_norm_host(x.data_ptr(), n, kind, C.byref(r)))
    return r.value


def bits(v):
    return np.float64(v).view(np.uint64)


@pytest.mark.parametrize("n", SIZES)
def test_reductions_on_integers_are_exact(n):
    """|x|, |y| <= 2^10, w in {1/4, 1/2, 1, 2}: every partial sum is an integer below 2^53, so exact in any order"""
    rng = rng_for(n, 6)
    xi, yi = rng.integers(-1024, 1025, n), rng.integers(-1024, 1025, n)
    w4 = rng.choice([1, 2, 4, 8], n)                    # 4 w
    x, y, w = xi.astype(np.float64), yi.astype(np.float64), w4 / 4.0
    d_x, d_y, d_w = dev(x, np.nan), dev(y, np.nan), dev(w, np.nan)
    exact_dot = float(int((xi * yi).sum()))
    exact_wdot = float(int((w4 * xi * yi).sum())) / 4.0
    assert bits(dot_dev(d_x, d_y, n)) == bits(exact_dot)
    assert bits(dot_host(d_x, d_y, n)) == bits(exact_dot)
    assert bits(dot_dev(d_x, d_y, n, d_w)) == bits(exact_wdot)
    assert bits(norm_host(d_x, n, 0)) == bits(float(int(np.abs(xi).sum())))
    assert bits(norm_host(d_x, n, 1)) == bits(math.sqrt(float(int((xi * xi).sum()))))
    assert bits(norm_host(d_x, n, 2)) == bits(float(np.abs(xi).max()) if n else 0.0)


@pytest.mark.parametrize("n", SIZES)
def test_reductions_on_random_data(n):
    """|got - fsum| <= (ceil(n / 151552) + 20) u sum|x_i y_i|; repeatable bit for bit; weighted = dot(w .* x, y)"""
    rng = rng_for(n, 7)
    x, y = randn(rng, n), randn(rng, n)
    w = 1.0 / rng.integers(1, 5, n)
    d_x, d_y, d_w = dev(x, np.nan), dev(y, np.nan), dev(w, np.nan)
    k = -(-n // RED_THREADS) + 20
    xy = x * y
    ref, scale = math.fsum(xy), math.fsum(np.abs(xy))
    got = dot_dev(d_x, d_y, n)
    assert abs(got - ref) <= k * U * scale, (got, ref)
    assert bits(dot_dev(d_x, d_y, n)) == bits(got)
    assert bits(dot_host(d_x, d_y, n)) == bits(got)
    wxy = (w * x) * y
    got_w = dot_dev(d_x, d_y, n, d_w)
    assert abs(got_w - math.fsum(wxy)) <= (k + 1) * U * math.fsum(np.abs(wxy))
    assert bits(dot_dev(d_x, d_y, n, d_w)) == bits(got_w)
    # solver.Vec.dot: (w .* a) . b in one pass rounds like pmult then dot
    wx = out(n)
    b2(lib.b200_vec_pointwise_mult(wx.data_ptr(), d_w.data_ptr(), d_x.data_ptr(), n))
    assert bits(dot_dev(wx, d_y, n)) == bits(got_w)
    # norms
    ax = np.abs(x)
    s1 = math.fsum(ax)
    got1 = norm_host(d_x, n, 0)
    assert abs(got1 - s1) <= k * U * s1
    s2 = math.fsum(x * x)
    got2 = norm_host(d_x, n, 1)
    assert abs(got2 - math.sqrt(s2)) <= (k / 2 + 2) * U * math.sqrt(s2)
    assert bits(norm_host(d_x, n, 1)) == bits(got2)
    assert bits(norm_host(d_x, n, 2)) == bits(float(ax.max()) if n else 0.0)


def oracle_max_norm(a):
    """oracle/ceed_cpu.c CeedVectorNorm, CEED_NORM_MAX: s = 0; s = |a_i| if |a_i| > s (NaN never compares greater)"""
    s = 0.0
    for v in a.tolist():
        if abs(v) > s:
            s = abs(v)
    return s


@pytest.mark.parametrize("case", ["nan_first", "all_nan", "inf_and_nan", "minus_inf", "sprinkled", "large"])
def test_max_norm_skips_nan_like_the_oracle(case):
    nan, inf = np.nan, np.inf
    rng = rng_for(8, case)
    x = {"nan_first": np.array([nan, 1.0, -3.0]), "all_nan": np.full(5, nan), "inf_and_nan": np.array([inf, nan, 2.0]),
         "minus_inf": np.array([nan, -inf, 2.0, nan]), "sprinkled": randn(rng, 1000),
         "large": randn(rng, VEC_THREADS + 1)}[case]
    if case in ("sprinkled", "large"):
        x[rng.choice(x.size, x.size // 10, replace=False)] = nan
        x[np.nanargmax(np.abs(x))] = nan      # the largest finite entry is NaN now: the max is the next one
    got = norm_host(dev(x, 1e308), x.size, 2)    # a read past the end would return the tail
    assert bits(got) == bits(oracle_max_norm(x))


# --------------------------------------------------------------------------- device-scalar Krylov steps

SCALARS = [0.0, -0.0, 1.0, -3.0, 1e-300, 1e300, np.inf, np.nan]


def krylov_steps(n, num, den, rng):
    """runs axpy_dev (both signs), aypx_dev and pcg_update (x given and NULL) on power-of-two vectors (exact products
    with any ratio), compares each bit for bit with the update by solver._guarded_ratio(num, den)"""
    a = _guarded_ratio(num, den)
    sc = dev(np.array([num, den]))
    p_num, p_den = sc.data_ptr(), sc.data_ptr() + 8
    x, y = pow2(rng, n), pow2(rng, n)
    d_x = dev(x, np.nan)
    for sign in (1.0, -1.0):
        d_y = dev(y, GUARD_VAL)
        b2(lib.b200_vec_axpy_dev(d_y.data_ptr(), d_x.data_ptr(), n, p_num, p_den, sign))
        assert_bits(fetch(d_y, n), y + (sign * a) * x, f"axpy_dev sign {sign} ({num}/{den})")
    d_y = dev(y, GUARD_VAL)
    b2(lib.b200_vec_aypx_dev(d_y.data_ptr(), d_x.data_ptr(), n, p_num, p_den))
    assert_bits(fetch(d_y, n), x + a * y, f"aypx_dev ({num}/{den})")
    r, p, Ap, dinv = pow2(rng, n), pow2(rng, n), pow2(rng, n), randn(rng, n)
    d_p, d_Ap, d_dinv = dev(p, np.nan), dev(Ap, np.nan), dev(dinv, np.nan)
    outs = []
    for with_x in (True, False):
        d_xx = dev(x, GUARD_VAL) if with_x else None
        d_r, d_z = dev(r, GUARD_VAL), out(n)
        b2(lib.b200_pcg_update(d_xx.data_ptr() if with_x else None, d_r.data_ptr(), d_z.data_ptr(), d_p.data_ptr(),
                               d_Ap.data_ptr(), d_dinv.data_ptr(), n, p_num, p_den))
        if with_x:
            assert_bits(fetch(d_xx, n), x + a * p, f"pcg_update x ({num}/{den})")
        outs.append((fetch(d_r, n), fetch(d_z, n)))
    rr = r - a * Ap
    assert_bits(outs[0][0], rr, f"pcg_update r ({num}/{den})")
    assert_bits(outs[0][1], dinv * rr, f"pcg_update z ({num}/{den})")
    assert_bits(outs[1][0], outs[0][0], "pcg_update r, x = NULL")
    assert_bits(outs[1][1], outs[0][1], "pcg_update z, x = NULL")


def test_device_scalar_steps_use_the_guarded_ratio():
    rng = rng_for(9)
    for num in SCALARS:
        for den in SCALARS:
            krylov_steps(4099, num, den, rng)


@pytest.mark.parametrize("n", SIZES)
def test_device_scalar_steps_over_the_sizes(n):
    krylov_steps(n, 3.0, -4.0, rng_for(n, 10))


# --------------------------------------------------------------------------- Chebyshev smoother


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("zero_guess", [0, 1])
def test_cheb_init_and_step_match_the_torch_branch(n, zero_guess):
    rng = rng_for(n, 11, zero_guess)
    x0, r0, d0, Ad, dinv = (randn(rng, n) for _ in range(5))
    inv_theta, c1, c2 = 1.0 / 1.37, 0.61, -0.23
    T = lambda a: torch.from_numpy(a.copy())
    # init, torch branch of ChebyshevJacobi.apply: d = dinv .* r; d *= 1/theta; x = d or x += d
    x_ref, d_ref = T(x0), torch.empty(n, dtype=torch.float64)
    torch.mul(T(dinv), T(r0), out=d_ref)
    d_ref.mul_(inv_theta)
    if zero_guess:
        x_ref.copy_(d_ref)
    else:
        x_ref.add_(d_ref)
    d_xx = out(n) if zero_guess else dev(x0, GUARD_VAL)    # zero_guess: x is not read, NaN must not leak in
    d_r, d_d, d_dinv = dev(r0, np.nan), out(n), dev(dinv, np.nan)
    b2(lib.b200_cheb_init(d_xx.data_ptr(), d_r.data_ptr(), d_d.data_ptr(), d_dinv.data_ptr(), inv_theta, zero_guess, n))
    assert_bits(fetch(d_d, n), d_ref.numpy(), "cheb_init d")
    if zero_guess:
        assert_bits(fetch(d_xx, n), x_ref.numpy(), "cheb_init x")
    else:
        assert_within(fetch(d_xx, n), x_ref.numpy(), np.abs(x0) + np.abs(d_ref.numpy()), 2, "cheb_init x")
    # step: r -= Ad; z = dinv .* r; d = c1 d + c2 z; x += d
    x_ref, r_ref, d_ref, z = T(x0), T(r0), T(d0), torch.empty(n, dtype=torch.float64)
    r_ref.sub_(T(Ad))
    torch.mul(T(dinv), r_ref, out=z)
    d_ref.mul_(c1).add_(z, alpha=c2)
    x_ref.add_(d_ref)
    d_xx, d_r, d_d = dev(x0, GUARD_VAL), dev(r0, GUARD_VAL), dev(d0, GUARD_VAL)
    b2(lib.b200_cheb_step(d_xx.data_ptr(), d_r.data_ptr(), d_d.data_ptr(), dev(Ad, np.nan).data_ptr(),
                          d_dinv.data_ptr(), c1, c2, n))
    assert_bits(fetch(d_r, n), r_ref.numpy(), "cheb_step r")
    d_scale = np.abs(c1 * d0) + np.abs(c2 * z.numpy())
    got_d = fetch(d_d, n)
    assert_within(got_d, d_ref.numpy(), d_scale, 4, "cheb_step d")
    assert_within(fetch(d_xx, n), x_ref.numpy(), np.abs(x0) + np.abs(got_d) + 2 * d_scale, 6, "cheb_step x")


@pytest.mark.parametrize("zero_guess", [False, True])
def test_chebyshev_apply_matches_the_torch_branch(zero_guess):
    n = VEC_THREADS + 1
    rng = rng_for(12, zero_guess)

    def A(x, y):   # 1-D Laplacian-like, the same torch statements on either device
        y.copy_(2.0 * x)
        y[1:] -= 0.5 * x[:-1]
        y[:-1] -= 0.5 * x[1:]

    b, x0, diag = rng.standard_normal(n), rng.standard_normal(n), 1.5 + rng.random(n)
    res = {}
    for device in ("cpu", "cuda"):
        s = ChebyshevJacobi(Vec(), A, n, device, its=3)
        s.dinv = torch.from_numpy(1.0 / diag).to(device)
        s.emin, s.emax = 0.2, 2.2
        x = torch.from_numpy(np.full(n, np.nan) if zero_guess else x0.copy()).to(device)
        s.apply(torch.from_numpy(b).to(device), x, zero_guess)
        res[device] = fetch(x)
    assert np.isfinite(res["cuda"]).all()
    assert np.abs(res["cuda"] - res["cpu"]).max() <= 1e-14 * np.abs(res["cpu"]).max()


# --------------------------------------------------------------------------- lattice transfers and 27-point stencil

LATTICES = [(2, 2, 2), (2, 3, 5), (4, 2, 3), (55, 55, 55)]   # 3 * 109^3 fine rows > one capped grid


def prolong(Nc, xc):
    Nf = [2 * v - 1 for v in Nc]
    nf = 3 * int(np.prod(Nf))
    f = out(nf)
    b2(lib.b200_lattice_prolong(*Nc, dev(xc, np.nan).data_ptr(), f.data_ptr()))
    return fetch(f, nf)


def restrict(Nc, xf):
    nc = 3 * int(np.prod(Nc))
    c = out(nc)
    b2(lib.b200_lattice_restrict(*Nc, dev(xf, np.nan).data_ptr(), c.data_ptr()))
    return fetch(c, nc)


@pytest.mark.parametrize("Nc", LATTICES, ids=str)
def test_lattice_transfers_match_the_cpu_branch(Nc):
    nc, nf = 3 * int(np.prod(Nc)), 3 * int(np.prod([2 * v - 1 for v in Nc]))
    rng = rng_for(13, *Nc)
    cpu_P = lambda v: _lattice_prolong_cpu(Nc, torch.from_numpy(v)).numpy()
    cpu_R = lambda v: _lattice_restrict_cpu(Nc, torch.from_numpy(v)).numpy()
    # dyadic: integers times the weights 1/2, 1/4, 1/8 are exact
    xc, xf = ints(rng, nc), ints(rng, nf)
    assert_bits(prolong(Nc, xc), cpu_P(xc), "prolong, integers")
    assert_bits(restrict(Nc, xf), cpu_R(xf), "restrict, integers")
    # random: at most 8 (prolong) / 27 (restrict) weighted terms
    xc, xf = randn(rng, nc), randn(rng, nf)
    assert_within(prolong(Nc, xc), cpu_P(xc), cpu_P(np.abs(xc)), 10, "prolong, random")
    assert_within(restrict(Nc, xf), cpu_R(xf), cpu_R(np.abs(xf)), 30, "restrict, random")
    # adjointness <P xc, xf> = <xc, R xf> (positive data: no cancellation)
    xc, xf = rng.random(nc), rng.random(nf)
    lhs, rhs = math.fsum(prolong(Nc, xc) * xf), math.fsum(xc * restrict(Nc, xf))
    assert abs(lhs - rhs) <= 1e-14 * max(lhs, rhs)


@pytest.mark.parametrize("Nc", LATTICES[:3], ids=str)
def test_lattice_restriction_is_the_transposed_prolongation(Nc):
    nc, nf = 3 * int(np.prod(Nc)), 3 * int(np.prod([2 * v - 1 for v in Nc]))
    Pm = np.stack([prolong(Nc, e) for e in np.eye(nc)], axis=1)
    Rm = np.stack([restrict(Nc, e) for e in np.eye(nf)], axis=1)
    assert_bits(Rm, Pm.T)
    cpu = np.stack([_lattice_prolong_cpu(Nc, torch.from_numpy(e)).numpy() for e in np.eye(nc)], axis=1)
    assert_bits(Pm, cpu)


def stencil_values(rng, N, gen):
    """(81, n) stencil values; entries that point outside the lattice are NaN (the kernel must not read them)"""
    n = 3 * int(np.prod(N))
    sv = gen(rng, 81 * n).reshape(81, n)
    i, j, k = lattice_ids(N)
    for o in range(27):
        dx, dy, dz = o % 3 - 1, (o // 3) % 3 - 1, o // 9 - 1
        bad = ~((i + dx >= 0) & (i + dx < N[0]) & (j + dy >= 0) & (j + dy < N[1]) & (k + dz >= 0) & (k + dz < N[2]))
        sv[o * 3:(o + 1) * 3, np.repeat(bad, 3)] = np.nan
    return sv


def stencil_spmv(N, sv, x):
    n = 3 * int(np.prod(N))
    y = out(n)
    b2(lib.b200_stencil27_spmv(*N, dev(sv).data_ptr(), dev(x, np.nan).data_ptr(), y.data_ptr()))
    return fetch(y, n)


@pytest.mark.parametrize("N", [(2, 2, 2), (3, 1, 4), (1, 4, 2), (4, 3, 5)], ids=str)
def test_stencil27_spmv_is_the_dense_matrix(N):
    rng = rng_for(14, *N)
    n = 3 * int(np.prod(N))
    sv = stencil_values(rng, N, lambda r, m: ints(r, m, 1024))
    x = ints(rng, n, 1024)
    A = dense_from_stencil(sv, N)
    assert_bits(stencil_spmv(N, sv, x), A @ x, "integers")
    sv = stencil_values(rng, N, randn)
    x = randn(rng, n)
    A = dense_from_stencil(sv, N)
    assert_within(stencil_spmv(N, sv, x), A @ x, np.abs(A) @ np.abs(x), 2 * 81 + 4, "random")


def test_stencil27_spmv_on_a_large_lattice_matches_scipy():
    """3 * 80 * 80 * 70 rows: several passes of the capped 128-thread grid; integers, so exact"""
    N = (80, 80, 70)
    n = 3 * int(np.prod(N))
    rng = rng_for(15)
    sv = rng.integers(-1024, 1025, (81, n), dtype=np.int16).astype(np.float64)
    x = ints(rng, n, 1024)
    i, j, k = lattice_ids(N)
    # CSR, row r = 3 node + a, slots (o, b) in stencil order; column 3 (node + dx + Nx (dy + Ny dz)) + b
    ok = np.empty((n // 3, 27), dtype=bool)
    col = np.empty((n // 3, 27), dtype=np.int64)
    for o in range(27):
        dx, dy, dz = o % 3 - 1, (o // 3) % 3 - 1, o // 9 - 1
        ok[:, o] = (i + dx >= 0) & (i + dx < N[0]) & (j + dy >= 0) & (j + dy < N[1]) & (k + dz >= 0) & (k + dz < N[2])
        col[:, o] = (i + dx) + N[0] * ((j + dy) + N[1] * (k + dz))
        sv[o * 3:(o + 1) * 3, np.repeat(~ok[:, o], 3)] = np.nan
    okr = np.repeat(np.repeat(ok, 3, axis=0)[:, :, None], 3, axis=2)                 # (n, 27, 3)
    ind = (3 * np.repeat(col, 3, axis=0)[:, :, None] + np.arange(3)).astype(np.int32)
    data = sv.reshape(27, 3, n).transpose(2, 0, 1)[okr]
    ind = ind[okr]
    indptr = np.concatenate([[0], np.cumsum(okr.reshape(n, -1).sum(axis=1))])
    A = sp.csr_matrix((data, ind, indptr), shape=(n, n))
    del data, ind, okr
    assert_bits(stencil_spmv(N, sv, x), A @ x)


# --------------------------------------------------------------------------- ELL mat-vec

ELL_CASES = [(n, s) for n in SIZES for s in (1, 27, 81) if 8 * n * s <= 1.0e9]


def ell_case(rng, n, nslots, gen):
    """slot-major cols/vals with random empty slots, whole empty rows and empty leading slots; vals of empty slots
    are NaN (never read)"""
    ncols = n // 2 + 1
    cols = rng.integers(0, ncols, (nslots, n)).astype(np.int32)
    cols[rng.random((nslots, n)) < 0.3] = -1
    r = np.arange(n)
    cols[:, r % 11 == 5] = -1                                         # empty rows
    lead = (r % 7 == 3)
    cols[:max(nslots - 1, 1), lead] = -1                              # empty leading slots
    vals = gen(rng, nslots * n).reshape(nslots, n)
    vals[cols < 0] = np.nan
    x = gen(rng, ncols)
    m = (cols >= 0).T
    A = sp.csr_matrix((vals.T[m], cols.T[m], np.concatenate([[0], np.cumsum(m.sum(axis=1))])), shape=(n, ncols))
    return cols, vals, x, A


def ell_spmv(n, nslots, cols, vals, x):
    y = out(n)
    b2(lib.b200_ell_spmv(n, nslots, dev(cols).data_ptr(), dev(vals).data_ptr(), dev(x, np.nan).data_ptr(),
                         y.data_ptr()))
    return fetch(y, n)


@pytest.mark.parametrize("n,nslots", ELL_CASES)
def test_ell_spmv_matches_scipy(n, nslots):
    rng = rng_for(n, nslots, 16)
    cols, vals, x, A = ell_case(rng, n, nslots, lambda r, m: ints(r, m, 1024))
    assert_bits(ell_spmv(n, nslots, cols, vals, x), A @ x)


@pytest.mark.parametrize("nslots", [1, 27, 81])
def test_ell_spmv_random_values(nslots):
    n = VEC_THREADS // 2 + 1
    rng = rng_for(nslots, 17)
    cols, vals, x, A = ell_case(rng, n, nslots, randn)
    Aabs = A.copy()
    Aabs.data = np.abs(Aabs.data)
    assert_within(ell_spmv(n, nslots, cols, vals, x), A @ x, Aabs @ np.abs(x), 2 * nslots + 4)


# --------------------------------------------------------------------------- ordered sums, bit for bit


def map_build(lsize, offsets):
    off = np.ascontiguousarray(offsets, dtype=np.int32)
    tptr = np.full(lsize + 1, -5, dtype=np.int32)
    tidx = np.full(max(off.size, 1), -5, dtype=np.int32)
    rc = lib.b200_transpose_map_build(lsize, off.size, off.ctypes.data, tptr.ctypes.data, tidx.ctypes.data)
    return rc, tptr, tidx[:off.size]


def ranks(groups):
    """(order, rank): positions sorted by group (stably) and the index of each inside its group"""
    order = np.argsort(groups, kind="stable")
    g = groups[order]
    return order, np.arange(g.size) - np.searchsorted(g, g, side="left")


def transpose_ref(L0, off, E, elemsize, ncomp, cs, layout):
    """L[o + c cs] += E-vector entries of the positions p with offsets[p] == o, one at a time, ascending p"""
    L = L0.copy()
    order, rank = ranks(off)
    for k in range(int(rank.max()) + 1 if rank.size else 0):
        p = order[rank == k]
        o = off[p].astype(np.int64)
        e, nn = p // elemsize, p % elemsize
        for c in range(ncomp):
            L[o + c * cs] += E[p * ncomp + c] if layout else E[(e * ncomp + c) * elemsize + nn]
    return L


def run_transpose(lsize, off, elemsize, ncomp, cs, layout, Lsize, rng):
    rc, tptr, tidx = map_build(lsize, off)
    assert rc == 0
    assert np.array_equal(tptr, np.concatenate([[0], np.cumsum(np.bincount(off, minlength=lsize))]))
    assert np.array_equal(tidx, np.argsort(off, kind="stable"))        # ascending positions within every offset
    L0, E = randn(rng, Lsize), randn(rng, off.size * ncomp)
    d_L = dev(L0, GUARD_VAL)
    b2(lib.b200_transpose_gather_add(lsize, dev(tptr).data_ptr(), dev(tidx, 0).data_ptr(), elemsize, ncomp, cs,
                                     layout, dev(E, np.nan).data_ptr(), d_L.data_ptr()))
    assert_bits(fetch(d_L, Lsize), transpose_ref(L0, off, E, elemsize, ncomp, cs, layout),
                f"layout {layout} ncomp {ncomp} compstride {cs}")


@pytest.mark.parametrize("layout", [0, 1])
def test_transpose_gather_add_on_a_box_mesh(layout):
    mesh = BoxMesh(n=(3, 4, 5), perturb=0.0, seed=0)
    rng = rng_for(18, layout)
    nn, es = mesh.num_nodes(2), 27
    node = mesh.offsets(2, ncomp=1).reshape(-1)
    run_transpose(nn, node, es, 1, 1, layout, nn, rng)
    run_transpose(nn, node, es, 1, nn, layout, nn, rng)
    run_transpose(nn, node, es, 3, nn, layout, 3 * nn, rng)                 # compstride = lsize
    run_transpose(3 * nn, mesh.offsets(2, ncomp=3).reshape(-1), es, 3, 1, layout, 3 * nn, rng)   # interleaved


@pytest.mark.parametrize("lsize", SIZES)
def test_transpose_gather_add_random_offsets(lsize):
    """random offsets leave some L entries unreferenced: those keep their value"""
    rng = rng_for(lsize, 19)
    es = 8
    npos = es * (lsize // es + 1) if lsize else 0
    off = rng.integers(0, max(lsize, 1), npos).astype(np.int32)
    for layout in (0, 1):
        run_transpose(lsize, off, es, 1, 1, layout, lsize, rng)
        run_transpose(lsize, off, es, 3, lsize, layout, 3 * lsize, rng)
    m = lsize // 3
    if m:
        run_transpose(3 * m, 3 * rng.integers(0, m, es * (m // es + 1)).astype(np.int32), es, 3, 1, 1, 3 * m, rng)


def test_transpose_map_build_refuses_out_of_range_offsets():
    for bad in (-1, 10):
        off = np.array([0, 3, bad, 9], dtype=np.int32)
        rc, _, _ = map_build(10, off)
        assert rc != 0
        assert "out of range" in lib.b200_last_error().decode()


def halo_case(rng, nuniq):
    """nuniq shared dofs with 2-8 holders each; the own entry (-1) first, in the middle or last"""
    ndof = nuniq + nuniq // 2 + 3
    udof = rng.permutation(ndof)[:nuniq].astype(np.int32)
    nh = rng.integers(2, 9, nuniq)
    uptr = np.concatenate([[0], np.cumsum(nh)]).astype(np.int32)
    u = np.arange(nuniq)
    own = np.where(u % 3 == 0, 0, np.where(u % 3 == 1, nh // 2, nh - 1))
    total = int(uptr[-1])
    nrecv = total - nuniq + 5
    uent = np.empty(total, dtype=np.int32)
    is_own = np.zeros(total, dtype=bool)
    is_own[uptr[:-1] + own] = True
    uent[is_own] = -1
    uent[~is_own] = rng.permutation(nrecv)[:total - nuniq]
    return ndof, udof, nh, uptr, uent, randn(rng, nrecv), randn(rng, ndof)


@pytest.mark.parametrize("nuniq", SIZES)
def test_halo_unpack_ordered_sums_in_holder_order(nuniq):
    rng = rng_for(nuniq, 20)
    ndof, udof, nh, uptr, uent, recv, y0 = halo_case(rng, nuniq)
    d_y = dev(y0, GUARD_VAL)
    b2(lib.b200_halo_unpack_ordered(nuniq, dev(udof).data_ptr(), dev(uptr).data_ptr(), dev(uent, 0).data_ptr(),
                                    dev(recv, np.nan).data_ptr(), d_y.data_ptr()))
    s = np.zeros(nuniq)
    for j in range(8):
        sel = np.flatnonzero(nh > j)
        ent = uent[uptr[sel] + j]
        s[sel] += np.where(ent < 0, y0[udof[sel]], recv[np.maximum(ent, 0)])
    ref = y0.copy()
    ref[udof] = s
    assert_bits(fetch(d_y, ndof), ref)


def assemble_elem_ref(ptr, src, evals, nblocks):
    """vals[k][i][j] = sum over t in [ptr[k], ptr[k+1]) of evals[src[t] + 24 j + i], in list order"""
    cnt = np.diff(ptr)
    blk = np.repeat(np.arange(nblocks), cnt)
    rank = np.arange(src.size) - np.repeat(ptr[:-1], cnt)
    vals = np.zeros((nblocks, 3, 3))
    ij = (24 * np.arange(3)[None, :] + np.arange(3)[:, None])        # [i][j] -> 24 j + i
    for k in range(int(rank.max()) + 1 if rank.size else 0):
        t = np.flatnonzero(rank == k)
        vals[blk[t]] += evals[src[t][:, None, None] + ij[None]]
    return vals.reshape(-1)


def run_assemble_elem(ptr, src, evals, nblocks):
    v = out(9 * nblocks)
    b2(lib.b200_bsr_assemble_elem(nblocks, dev(ptr).data_ptr(), dev(src, 0).data_ptr(), dev(evals).data_ptr(),
                                  v.data_ptr()))
    assert_bits(fetch(v, 9 * nblocks), assemble_elem_ref(ptr, src, evals, nblocks))


def test_bsr_assemble_elem_on_tube_element_matrices():
    m = tube_mesh(2, 8, 3)
    en = m.offsets(1).reshape(-1, 8).astype(np.int64) // 3
    nn, E = m.num_nodes(1), en.shape[0]
    a_, b_ = np.meshgrid(np.arange(8), np.arange(8), indexing="ij")
    a_, b_ = a_.reshape(-1), b_.reshape(-1)
    key = (en[:, a_] * nn + en[:, b_]).reshape(-1)
    src = ((np.arange(E)[:, None] * 24 + 3 * b_[None]) * 24 + 3 * a_[None]).reshape(-1)
    keys, dest = np.unique(key, return_inverse=True)
    order = np.argsort(dest, kind="stable")
    ptr = np.concatenate([[0], np.cumsum(np.bincount(dest, minlength=keys.size))]).astype(np.int64)
    run_assemble_elem(ptr, src[order].astype(np.int64), randn(rng_for(21), E * 576), keys.size)


@pytest.mark.parametrize("nblocks", [0, 1, 257, RED_THREADS + 1])
def test_bsr_assemble_elem_with_empty_ranges(nblocks):
    rng = rng_for(nblocks, 22)
    E = 50
    cnt = rng.integers(0, 5, nblocks)
    cnt[::3] = 0
    ptr = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
    nt = int(ptr[-1])
    src = ((rng.integers(0, E, nt) * 24 + 3 * rng.integers(0, 8, nt)) * 24 + 3 * rng.integers(0, 8, nt)).astype(np.int64)
    run_assemble_elem(ptr, src, randn(rng, E * 576), nblocks)


# --------------------------------------------------------------------------- AMG block kernels against scipy

BSR_SHAPES = [(3, 3), (6, 6), (3, 6), (6, 3)]
PAIR_SHAPES = [(3, 3, 6), (6, 3, 6), (6, 6, 6), (3, 3, 3)]


def bsr_case(rng, nbrows, br, bc, gen):
    """rows of 0, 1, 40-60 and 2-10 blocks in turn, sorted distinct columns"""
    ncols = 97
    lens = np.select([np.arange(nbrows) % 4 == k for k in range(3)],
                     [0, 1, rng.integers(40, 61, nbrows)], rng.integers(2, 11, nbrows))
    rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    colidx = np.concatenate([np.sort(rng.choice(ncols, L, replace=False)) for L in lens] + [np.zeros(0, int)])
    vals = gen(rng, int(rowptr[-1]) * br * bc)
    x = gen(rng, ncols * bc)
    A = sp.bsr_matrix((vals.reshape(-1, br, bc), colidx.astype(np.int32), rowptr), shape=(nbrows * br, ncols * bc))
    return rowptr, colidx.astype(np.int32), vals, x, A, lens


def bsr_spmv(br, bc, nbrows, rowptr, colidx, vals, x):
    y = out(nbrows * br)
    b2(lib.b200_bsr_spmv(br, bc, nbrows, dev(rowptr).data_ptr(), dev(colidx, 0).data_ptr(), dev(vals).data_ptr(),
                         dev(x, np.nan).data_ptr(), y.data_ptr()))
    return fetch(y, nbrows * br)


@pytest.mark.parametrize("br,bc", BSR_SHAPES)
@pytest.mark.parametrize("nbrows", [0, 1, 3, 203])
def test_bsr_spmv_matches_scipy(br, bc, nbrows):
    rng = rng_for(br, bc, nbrows, 23)
    rowptr, colidx, vals, x, A, lens = bsr_case(rng, nbrows, br, bc, lambda r, m: ints(r, m, 1024))
    assert_bits(bsr_spmv(br, bc, nbrows, rowptr, colidx, vals, x), A @ x if nbrows else np.zeros(0), "integers")
    rowptr, colidx, vals, x, A, lens = bsr_case(rng, nbrows, br, bc, randn)
    if nbrows:
        terms = np.repeat(lens * bc, br)
        assert_within(bsr_spmv(br, bc, nbrows, rowptr, colidx, vals, x), A @ x, abs(A) @ np.abs(x), 2 * terms + 16,
                      "random")


def pairs_case(rng, shape, nout, gen):
    br, bk, bc = shape
    nA, nB, nT, nrow = 50, 60, 40, 30
    cnt = rng.integers(0, 6, nout)
    cnt[::4] = 0
    ptr = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int64)
    nt = int(ptr[-1])
    pa, pb = rng.integers(0, nA, nt).astype(np.int32), rng.integers(0, nB, nt).astype(np.int32)
    A, B = gen(rng, nA * br * bk), gen(rng, nB * bk * bc)
    tmap = rng.integers(0, nT, nout).astype(np.int32)
    tmap[rng.random(nout) < 0.3] = -1
    rowof = rng.integers(0, nrow, nout).astype(np.int32)
    T = gen(rng, nT * br * bc)
    dinv = rng.integers(1, 64, nrow * br) / 16.0
    return ptr, pa, pb, A, B, tmap, rowof, T, dinv


def pairs_ref(shape, ptr, pa, pb, A, B, tmap=None, rowof=None, T=None, dinv=None, omega=None):
    br, bk, bc = shape
    nout = ptr.size - 1
    Ab, Bb = A.reshape(-1, br, bk), B.reshape(-1, bk, bc)
    cnt = np.diff(ptr)
    k_of = np.repeat(np.arange(nout), cnt)
    rank = np.arange(pa.size) - np.repeat(ptr[:-1], cnt)
    Cm = np.zeros((nout, br, bc))
    for r in range(int(rank.max()) + 1 if rank.size else 0):
        t = np.flatnonzero(rank == r)
        Cm[k_of[t]] += Ab[pa[t]] @ Bb[pb[t]]
    if tmap is not None:
        T0 = np.where((tmap >= 0)[:, None, None], T.reshape(-1, br, bc)[np.maximum(tmap, 0)], 0.0)
        f = omega * dinv.reshape(-1, br)[rowof][:, :, None]
        Cm = T0 - f * Cm
    return Cm.reshape(-1)


def pairs_run(shape, ptr, pa, pb, A, B, epi, tmap, rowof, T, dinv, omega):
    br, bk, bc = shape
    nout = ptr.size - 1
    Cd = out(nout * br * bc)
    ptrs = [dev(tmap).data_ptr(), dev(rowof).data_ptr(), dev(T).data_ptr(), dev(dinv).data_ptr(),
            dev(np.array([omega])).data_ptr()] if epi else [None] * 5
    b2(lib.b200_bsr_pairs_product(br, bk, bc, nout, dev(ptr).data_ptr(), dev(pa, 0).data_ptr(), dev(pb, 0).data_ptr(),
                                  dev(A).data_ptr(), dev(B).data_ptr(), Cd.data_ptr(), *ptrs))
    return fetch(Cd, nout * br * bc)


@pytest.mark.parametrize("shape", PAIR_SHAPES, ids=str)
@pytest.mark.parametrize("epi", [False, True], ids=["plain", "epilogue"])
@pytest.mark.parametrize("nout", [0, 1, 300])
def test_bsr_pairs_product_matches_the_list_order_sum(shape, epi, nout):
    rng = rng_for(*shape, epi, nout, 24)
    omega = 0.75
    ptr, pa, pb, A, B, tmap, rowof, T, dinv = pairs_case(rng, shape, nout, lambda r, m: ints(r, m, 256))
    got = pairs_run(shape, ptr, pa, pb, A, B, epi, tmap, rowof, T, dinv, omega)
    ref = pairs_ref(shape, ptr, pa, pb, A, B, *((tmap, rowof, T, dinv, omega) if epi else ()))
    assert_bits(got, ref, "integers")
    ptr, pa, pb, A, B, tmap, rowof, T, dinv = pairs_case(rng, shape, nout, randn)
    omega = 0.6180339887498949
    got = pairs_run(shape, ptr, pa, pb, A, B, epi, tmap, rowof, T, dinv, omega)
    ref = pairs_ref(shape, ptr, pa, pb, A, B, *((tmap, rowof, T, dinv, omega) if epi else ()))
    scale = pairs_ref(shape, ptr, pa, pb, np.abs(A), np.abs(B))
    if epi:
        br, bk, bc = shape
        T0 = np.where((tmap >= 0)[:, None, None], np.abs(T).reshape(-1, br, bc)[np.maximum(tmap, 0)], 0.0)
        scale = (T0 + omega * dinv.reshape(-1, br)[rowof][:, :, None] * scale.reshape(-1, br, bc)).reshape(-1)
    terms = np.repeat(np.diff(ptr) * shape[1], shape[0] * shape[2])
    assert_within(got, ref, scale, 2 * terms + 8, "random")


@pytest.mark.parametrize("br,bc", [(3, 6), (6, 6), (3, 3)])
@pytest.mark.parametrize("nblocks", [0, 1, 257, 100003])
def test_bsr_transpose_gather(br, bc, nblocks):
    rng = rng_for(br, bc, nblocks, 25)
    nsrc = nblocks // 2 + 3
    src = randn(rng, nsrc * br * bc)
    idx = rng.integers(0, nsrc, nblocks).astype(np.int32)
    dst = out(nblocks * br * bc)
    b2(lib.b200_bsr_transpose_gather(br, bc, nblocks, dev(idx, 0).data_ptr(), dev(src).data_ptr(), dst.data_ptr()))
    assert_bits(fetch(dst, nblocks * br * bc), src.reshape(-1, br, bc)[idx].transpose(0, 2, 1).reshape(-1))


def test_block_shapes_that_are_not_instantiated_are_refused():
    """checked on the host before any launch"""
    z_i, z_l, z_d = dev(np.zeros(64, np.int32)), dev(np.zeros(64, np.int64)), dev(np.zeros(64 * 36))
    for br, bc in ((4, 4), (3, 4), (6, 9), (1, 1)):
        assert lib.b200_bsr_spmv(br, bc, 1, z_i.data_ptr(), z_i.data_ptr(), z_d.data_ptr(), z_d.data_ptr(),
                                 z_d.data_ptr()) != 0
        assert "not instantiated" in lib.b200_last_error().decode()
    for br, bk, bc in ((3, 6, 6), (6, 6, 3), (6, 3, 3), (3, 6, 3)):
        assert lib.b200_bsr_pairs_product(br, bk, bc, 1, z_l.data_ptr(), z_i.data_ptr(), z_i.data_ptr(), z_d.data_ptr(),
                                          z_d.data_ptr(), z_d.data_ptr(), None, None, None, None, None) != 0
        assert "not instantiated" in lib.b200_last_error().decode()
    assert lib.b200_bsr_pairs_product(3, 3, 6, 1, z_l.data_ptr(), z_i.data_ptr(), z_i.data_ptr(), z_d.data_ptr(),
                                      z_d.data_ptr(), z_d.data_ptr(), z_i.data_ptr(), None, z_d.data_ptr(),
                                      z_d.data_ptr(), z_d.data_ptr()) != 0
    assert "epilogue" in lib.b200_last_error().decode()
    for br, bc in ((6, 3), (3, 4)):
        assert lib.b200_bsr_transpose_gather(br, bc, 1, z_i.data_ptr(), z_d.data_ptr(), z_d.data_ptr()) != 0
        assert "not instantiated" in lib.b200_last_error().decode()
    torch.cuda.synchronize()
