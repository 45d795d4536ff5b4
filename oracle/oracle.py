"""TEST INFRASTRUCTURE ONLY -- see oracle/README.md.

ctypes loader for the CPU oracle (oracle/liboracle.so = ceed_oracle.c + qf_port.c)
and, when it has been built, the reference's own QFunctions
(oracle/_ref/libref_qf.so, compiled from /root/reference/qfunctions by oracle/Makefile).

May be imported only by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package never imports it.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_REF = None
_NATIVE = None
_REF_FAST = None

QFN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.POINTER(C.POINTER(C.c_double)),
                  C.POINTER(C.POINTER(C.c_double)))

QF_NAMES = ["SetupGeo", "LinElasF", "LinElasdF", "HyperSSF", "HyperSSdF", "HyperFSF", "HyperFSdF"]
PROBLEMS = {
    "linElas": ("LinElasF", "LinElasdF", False),
    "hyperSS": ("HyperSSF", "HyperSSdF", True),
    "hyperFS": ("HyperFSF", "HyperFSdF", True),
}


class Physics(C.Structure):
    """elasticity.h:30-37 Physics_private"""
    _fields_ = [("nu", C.c_double), ("E", C.c_double)]


def build(force=False):
    so = os.path.join(HERE, "liboracle.so")
    srcs = [os.path.join(HERE, f) for f in ("ceed_oracle.c", "qf_port.c", "ref_qf.c", "Makefile")]
    stale = force or not os.path.exists(so) or any(
        os.path.getmtime(s) > os.path.getmtime(so) for s in srcs if os.path.exists(s))
    ref_so = os.path.join(HERE, "_ref", "libref_qf.so")
    if os.path.isdir("/root/reference/qfunctions") and not os.path.exists(ref_so):
        stale = True
    if stale:
        subprocess.run(["make", "-s", "-C", HERE], check=True, stdout=subprocess.DEVNULL)
    return so


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
    return _LIB


def native_lib():
    """TIMING build (-O3 -march=native, FP contraction on), compiled on the box that runs it: bench.py's CPU legs only.
    Built in a temporary directory that is gone once the library is loaded: the benchmark writes nothing into the tree.
    Parity checks always go through lib()."""
    global _NATIVE
    if _NATIVE is None:
        with tempfile.TemporaryDirectory(prefix="oracle_native_") as d:
            subprocess.run(["make", "-s", "-C", HERE, "timing", "NATIVE_DIR=" + d], check=True, stdout=subprocess.DEVNULL)
            _NATIVE = C.CDLL(os.path.join(d, "liboracle_native.so"))
    return _NATIVE


def have_ref():
    return os.path.exists(os.path.join(HERE, "_ref", "libref_qf.so"))


def ref():
    global _REF
    if _REF is None:
        lib()
        _REF = C.CDLL(os.path.join(HERE, "_ref", "libref_qf.so"))
    return _REF


def have_ref_fast():
    return os.path.exists(os.path.join(HERE, "_ref", "libref_qf_fast.so"))


def ref_fast():
    """The reference's QFunctions at -O3 -march=x86-64-v3 (timing legs only)."""
    global _REF_FAST
    if _REF_FAST is None:
        _REF_FAST = C.CDLL(os.path.join(HERE, "_ref", "libref_qf_fast.so"))
    return _REF_FAST


def qf(name, which="port"):
    """Function pointer (as c_void_p-castable) of a QFunction; which in {port, ref, ref_fast, port_native}."""
    if which == "ref":
        return C.cast(getattr(ref(), "ref_" + name), C.c_void_p)
    if which == "ref_fast":
        return C.cast(getattr(ref_fast(), "ref_" + name), C.c_void_p)
    if which == "port_native":
        return C.cast(getattr(native_lib(), "port_" + name), C.c_void_p)
    return C.cast(getattr(lib(), "port_" + name), C.c_void_p)


def default_which():
    return "ref" if have_ref() else "port"


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def call_qf(name, which, ctx, Q, ins, nouts_sizes):
    """Call a QFunction on host arrays: ins = list of [size][Q] arrays."""
    ins = [_f64(a) for a in ins]
    outs = [np.zeros((s, Q)) for s in nouts_sizes]
    inp = (C.POINTER(C.c_double) * len(ins))(*[a.ctypes.data_as(C.POINTER(C.c_double)) for a in ins])
    outp = (C.POINTER(C.c_double) * len(outs))(*[a.ctypes.data_as(C.POINTER(C.c_double)) for a in outs])
    f = C.cast(qf(name, which), QFN)
    ctxp = C.cast(C.pointer(ctx), C.c_void_p) if ctx is not None else None
    rc = f(ctxp, Q, inp, outp)
    assert rc == 0
    return outs


def gauss(Q):
    x, w = np.zeros(Q), np.zeros(Q)
    lib().oracle_gauss(Q, _p(x), _p(w))
    return x, w


def lobatto(Q):
    x, w = np.zeros(Q), np.zeros(Q)
    lib().oracle_lobatto(Q, _p(x), _p(w))
    return x, w


def basis_1d(P, Q, qmode=0):
    """(interp1d[Q,P], grad1d[Q,P], qref1d[Q], qweight1d[Q]); qmode 0 Gauss, 1 Lobatto."""
    B, D, qr, qw = np.zeros((Q, P)), np.zeros((Q, P)), np.zeros(Q), np.zeros(Q)
    lib().oracle_basis_1d(P, Q, qmode, _p(B), _p(D), _p(qr), _p(qw))
    return B, D, qr, qw


def basis_apply(nelem, ncomp, P, Q, B, D, qw, tmode, emode, u):
    P3, Q3 = P ** 3, Q ** 3
    u = _f64(u) if u is not None else None
    if emode == 4:
        v = np.zeros((nelem, Q3))
    elif not tmode:
        v = np.zeros((nelem, 3 * ncomp * Q3 if emode == 2 else ncomp * Q3))
    else:
        v = np.zeros((nelem, ncomp * P3))
    rc = lib().oracle_basis_apply(nelem, ncomp, P, Q, _p(_f64(B)), _p(_f64(D)),
                                  _p(_f64(qw)) if qw is not None else None, int(tmode), emode,
                                  _p(u), _p(v))
    assert rc == 0
    return v


def setup_geo(nelem, Q, xoffsets, xcoord, which=None):
    which = which or default_which()
    qdata = np.zeros((nelem, 10, Q ** 3))
    rc = lib().oracle_setup_geo(qf("SetupGeo", which), nelem, Q, _p(_i32(xoffsets)),
                                _p(_f64(xcoord)), _p(qdata))
    assert rc == 0
    return qdata


def operator_apply(problem, jacobian, phys, nelem, P, Q, B, D, offsets, qdata, gradu, x,
                   which=None, y=None, native=False):
    """y = A_loc x (zeroed first, CeedOperatorApply semantics).  Residual writes gradu.
    native=True runs the -march=native timing build of the operator loop (bench.py CPU legs)."""
    which = which or default_which()
    L = native_lib() if native else lib()
    fname, dfname, has_gradu = PROBLEMS[problem]
    mode = 0 if not has_gradu else (2 if jacobian else 1)
    x = _f64(x)
    if y is None:
        y = np.zeros_like(x)
    else:
        y[...] = 0
    ctx = Physics(*phys)
    rc = L.oracle_operator_apply_add(
        qf(dfname if jacobian else fname, which), C.byref(ctx), mode, nelem, P, Q, _p(_f64(B)),
        _p(_f64(D)), _p(_i32(offsets)), _p(qdata), _p(gradu) if has_gradu else None, _p(x), _p(y))
    assert rc == 0
    return y


def operator_diagonal(problem, phys, nelem, P, Q, B, D, offsets, qdata, gradu, lsize, which=None):
    which = which or default_which()
    _, dfname, has_gradu = PROBLEMS[problem]
    diag = np.zeros(lsize)
    ctx = Physics(*phys)
    rc = lib().oracle_operator_diagonal_add(
        qf(dfname, which), C.byref(ctx), 2 if has_gradu else 0, nelem, P, Q, _p(_f64(B)), _p(_f64(D)),
        _p(_i32(offsets)), _p(qdata), _p(gradu) if has_gradu else None, _p(diag))
    assert rc == 0
    return diag


def multiplicity(nelem, elemsize, ncomp, lsize, offsets):
    m = np.zeros(lsize)
    lib().oracle_multiplicity(nelem, elemsize, ncomp, 1, lsize, _p(_i32(offsets)), _p(m))
    return m


def transfer(transpose, nelem, Pc, Pf, offc, offf, vin, lsize_out):
    Bcf, _, _, _ = basis_1d(Pc, Pf, 1)
    out = np.zeros(lsize_out)
    rc = lib().oracle_transfer_add(int(transpose), nelem, Pc, Pf, _p(Bcf), _p(_i32(offc)),
                                   _p(_i32(offf)), _p(_f64(vin)), _p(out))
    assert rc == 0
    return out


def num_threads(native=False):
    return (native_lib() if native else lib()).oracle_num_threads()


def set_num_threads(n, native=False):
    """OpenMP threads of the oracle's element loops (torchrun exports OMP_NUM_THREADS=1 to its workers)."""
    return (native_lib() if native else lib()).oracle_set_num_threads(int(n))
