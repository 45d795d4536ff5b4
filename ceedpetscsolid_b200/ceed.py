"""ctypes binding of libceed_b200.so: the libCEED user API served by the `/gpu/b200` backend
(include/ceed/ceed.h) plus the thin C-ABI CUDA layer (include/b200_kernels.h).

Thin object wrappers with libCEED's own vocabulary (Ceed, Vector, ElemRestriction, Basis,
QFunction, Operator); argument order and meaning follow the C API the reference calls
(/root/reference/src/setuplibceed.c, src/matops.c).  Device arrays are torch CUDA tensors
(float64), borrowed zero-copy with CEED_USE_POINTER exactly as the reference borrows PETSc
VecCUDA arrays (matops.c:37-41).

The library is REQUIRED: importing this module without a built libceed_b200.so raises.
There is no Python / CPU fallback path.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIBPATH = os.environ.get("CEED_B200_LIB", os.path.join(HERE, "libceed_b200.so"))  # override: tuning builds only

MEM_HOST, MEM_DEVICE = 0, 1
COPY_VALUES, USE_POINTER, OWN_POINTER = 0, 1, 2
NOTRANSPOSE, TRANSPOSE = 0, 1
EVAL_NONE, EVAL_INTERP, EVAL_GRAD, EVAL_DIV, EVAL_CURL, EVAL_WEIGHT = 0, 1, 2, 4, 8, 16
GAUSS, GAUSS_LOBATTO = 0, 1
NORM_1, NORM_2, NORM_MAX = 0, 1, 2
PROBLEMS = {"linElas": 0, "hyperSS": 1, "hyperFS": 2}


class CeedError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIBPATH):
        raise ImportError(
            f"{LIBPATH} is missing: build it with `make -C ceedpetscsolid_b200/csrc` "
            "(or `python -c 'import __graft_entry__ as g; g.build()'`). The /gpu/b200 backend has no fallback.")
    return C.CDLL(LIBPATH, mode=C.RTLD_GLOBAL)


lib = _load()

_vp, _i, _d, _sz, _ll = C.c_void_p, C.c_int, C.c_double, C.c_size_t, C.c_longlong
_pvp = C.POINTER(C.c_void_p)


def _proto(name, *argtypes, restype=C.c_int):
    f = getattr(lib, name)
    f.argtypes = list(argtypes)
    f.restype = restype
    return f


# ---- libCEED API ------------------------------------------------------------------------
_proto("CeedInit", C.c_char_p, _pvp)
_proto("CeedDestroy", _pvp)
_proto("CeedGetResource", _vp, C.POINTER(C.c_char_p))
_proto("CeedGetPreferredMemType", _vp, C.POINTER(_i))
_proto("CeedSetErrorHandler", _vp, _vp)
_proto("CeedGetErrorMessage", _vp, C.POINTER(C.c_char_p))
_proto("CeedVectorCreate", _vp, _i, _pvp)
_proto("CeedVectorSetArray", _vp, _i, _i, _vp)
_proto("CeedVectorTakeArray", _vp, _i, _pvp)
_proto("CeedVectorSetValue", _vp, _d)
_proto("CeedVectorSyncArray", _vp, _i)
_proto("CeedVectorGetArray", _vp, _i, _pvp)
_proto("CeedVectorGetArrayRead", _vp, _i, _pvp)
_proto("CeedVectorRestoreArray", _vp, _pvp)
_proto("CeedVectorRestoreArrayRead", _vp, _pvp)
_proto("CeedVectorNorm", _vp, _i, C.POINTER(_d))
_proto("CeedVectorReciprocal", _vp)
_proto("CeedVectorGetLength", _vp, C.POINTER(_i))
_proto("CeedVectorDestroy", _pvp)
_proto("CeedElemRestrictionCreate", _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _pvp)
_proto("CeedElemRestrictionCreateStrided", _vp, _i, _i, _i, _i, _vp, _pvp)
_proto("CeedElemRestrictionCreateVector", _vp, _pvp, _pvp)
_proto("CeedElemRestrictionApply", _vp, _i, _vp, _vp, _vp)
_proto("CeedElemRestrictionGetMultiplicity", _vp, _vp)
_proto("CeedElemRestrictionDestroy", _pvp)
_proto("CeedBasisCreateTensorH1Lagrange", _vp, _i, _i, _i, _i, _i, _pvp)
_proto("CeedBasisCreateTensorH1", _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _pvp)
_proto("CeedBasisApply", _vp, _i, _i, _i, _vp, _vp)
_proto("CeedBasisGetNumQuadraturePoints", _vp, C.POINTER(_i))
_proto("CeedBasisGetInterp1D", _vp, _pvp)
_proto("CeedBasisGetGrad1D", _vp, _pvp)
_proto("CeedBasisGetQRef", _vp, _pvp)
_proto("CeedBasisGetQWeights", _vp, _pvp)
_proto("CeedBasisDestroy", _pvp)
_proto("CeedQFunctionCreateInterior", _vp, _i, _vp, C.c_char_p, _pvp)
_proto("CeedQFunctionCreateIdentity", _vp, _i, _i, _i, _pvp)
_proto("CeedQFunctionAddInput", _vp, C.c_char_p, _i, _i)
_proto("CeedQFunctionAddOutput", _vp, C.c_char_p, _i, _i)
_proto("CeedQFunctionSetContext", _vp, _vp, _sz)
_proto("CeedQFunctionDestroy", _pvp)
_proto("CeedOperatorCreate", _vp, _vp, _vp, _vp, _pvp)
_proto("CeedCompositeOperatorCreate", _vp, _pvp)
_proto("CeedCompositeOperatorAddSub", _vp, _vp)
_proto("CeedOperatorSetField", _vp, C.c_char_p, _vp, _vp, _vp)
_proto("CeedOperatorApply", _vp, _vp, _vp, _vp)
_proto("CeedOperatorApplyAdd", _vp, _vp, _vp, _vp)
_proto("CeedOperatorLinearAssembleDiagonal", _vp, _vp, _vp)
_proto("CeedOperatorLinearAssembleAddDiagonal", _vp, _vp, _vp)
_proto("CeedOperatorLinearAssembleSymbolic", _vp, C.POINTER(_i), C.POINTER(C.POINTER(_i)), C.POINTER(C.POINTER(_i)))
_proto("CeedOperatorLinearAssemble", _vp, _vp)
_proto("CeedOperatorDestroy", _pvp)
_proto("CeedOperatorIsFusedB200", _vp, C.POINTER(_i))
_proto("CeedOperatorIsJitFusedB200", _vp, C.POINTER(_i))
_proto("CeedOperatorApplyAddRangeB200", _vp, _vp, _vp, _i, _i)
_proto("CeedOperatorSetTransferScalingB200", _vp, _vp, _i)
_proto("CeedOperatorApplyPartitionedB200", _vp, _vp, _vp, _i, _vp, _vp, _i)
_proto("CeedIsDeterministic", _vp, _vp)
_proto("CeedB200LaunchCount", restype=C.c_ulonglong)
_proto("CeedB200LaunchCountReset", restype=None)
_proto("CeedB200SetStream", _vp, _vp)
_proto("CeedB200Synchronize", _vp)

# ---- thin CUDA layer (used by the harness: vector ops, maps, halos) -----------------------
_proto("b200_last_error", restype=C.c_char_p)
_proto("b200_set_device", _i)
_proto("b200_set_stream", _vp)
_proto("b200_sync")
_proto("b200_device_name", C.c_char_p, _i)
_proto("b200_launch_count", restype=C.c_ulonglong)
_proto("b200_launch_count_reset", restype=None)
_proto("b200_vec_set", _vp, _d, _sz)
_proto("b200_vec_scale", _vp, _d, _sz)
_proto("b200_vec_axpy", _vp, _d, _vp, _sz)
_proto("b200_vec_aypx", _vp, _d, _vp, _sz)
_proto("b200_vec_axpby", _vp, _d, _vp, _d, _vp, _sz)
_proto("b200_vec_pointwise_mult", _vp, _vp, _vp, _sz)
_proto("b200_vec_dot", _vp, _vp, _sz, _vp)
_proto("b200_vec_dot_weighted", _vp, _vp, _vp, _sz, _vp)
_proto("b200_vec_dot_host", _vp, _vp, _sz, C.POINTER(_d))
_proto("b200_vec_norm_host", _vp, _sz, _i, C.POINTER(_d))
_proto("b200_gather", _vp, _vp, _vp, _sz)
_proto("b200_scatter_set", _vp, _vp, _vp, _sz)
_proto("b200_scatter_add", _vp, _vp, _vp, _sz)
_proto("b200_mask_zero", _vp, _vp, _sz)
_proto("b200_gather_or_zero", _vp, _vp, _vp, _sz)
_proto("b200_copy_where", _vp, _vp, _vp, _sz)
_proto("b200_ell_spmv", _sz, _i, _vp, _vp, _vp, _vp)
_proto("b200_vec_axpy_dev", _vp, _vp, _sz, _vp, _vp, _d)
_proto("b200_vec_aypx_dev", _vp, _vp, _sz, _vp, _vp)
_proto("b200_pcg_update", _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _vp)
_proto("b200_stencil27_spmv", _i, _i, _i, _vp, _vp, _vp)
_proto("b200_stencil27_galerkin", _i, _i, _i, _vp, _vp)
_proto("b200_fp64_probe", C.POINTER(_d))
_proto("b200_ipc_get_handle", _vp, _vp)
_proto("b200_ipc_open", _vp, _pvp)
_proto("b200_ipc_close", _vp)
_proto("b200_halo_window_bytes", _sz, restype=_sz)
_proto("b200_halo_create", _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _i, _vp, _vp, _vp, _d, _pvp)
_proto("b200_halo_destroy", _vp)
_proto("b200_halo_begin", _vp, _vp)
_proto("b200_halo_end", _vp, _vp)
_proto("b200_halo_error", _vp, _vp)
_proto("b200_halo_unpack_ordered", _i, _vp, _vp, _vp, _vp, _vp)
_proto("b200_lattice_prolong", _i, _i, _i, _vp, _vp)
_proto("b200_lattice_restrict", _i, _i, _i, _vp, _vp)
_proto("b200_cheb_init", _vp, _vp, _vp, _vp, _d, _i, _sz)
_proto("b200_cheb_step", _vp, _vp, _vp, _vp, _vp, _d, _d, _sz)
_proto("b200_vec_reciprocal", _vp, _sz)
_proto("b200_elems_per_block", _i)
_proto("b200_fused_supported", _i, _i)
_proto("b200_jcache_ncomp", _i)
_proto("b200_apply_transfer", _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp)
_proto("b200_bsr_spmv", _i, _i, _i, _vp, _vp, _vp, _vp, _vp)
_proto("b200_bsr_pairs_product", _i, _i, _i, _sz, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp)
_proto("b200_bsr_transpose_gather", _i, _i, _sz, _vp, _vp, _vp)
_proto("b200_bsr_assemble_elem", _sz, _vp, _vp, _vp, _vp)
_proto("b200_jit_read_source", C.c_char_p, _pvp, C.c_char_p, _sz)
_proto("b200_jit_free_source", _vp, restype=None)
_proto("b200_jit_compile", _vp, C.c_char_p, C.c_char_p, _i, _vp, _i, _vp, C.POINTER(_i))
_proto("b200_jit_program", _i, restype=C.c_char_p)
_proto("b200_jit_fused_compile", _vp, C.c_char_p, C.c_char_p, _i, _vp, _i, _vp, _i, _i, _i, _i, C.POINTER(_i))
_proto("b200_jit_assemble_compile", _vp, C.c_char_p, C.c_char_p, _i, _vp, _i, _vp, _i, _i, _i, _i, C.POINTER(_i))
_proto("b200_jit_assemble_apply", _i, _vp, _sz, _i, _vp, _vp, _i, _vp, _vp)
_proto("b200_jit_compile_count", restype=C.c_ulonglong)

# sentinels are exported data symbols holding pointers
def _sentinel(name):
    return C.c_void_p.in_dll(lib, name).value


BASIS_COLLOCATED = _sentinel("CEED_BASIS_COLLOCATED")
VECTOR_ACTIVE = _sentinel("CEED_VECTOR_ACTIVE")
VECTOR_NONE = _sentinel("CEED_VECTOR_NONE")
ELEMRESTRICTION_NONE = _sentinel("CEED_ELEMRESTRICTION_NONE")
QFUNCTION_NONE = _sentinel("CEED_QFUNCTION_NONE")
REQUEST_IMMEDIATE = _sentinel("CEED_REQUEST_IMMEDIATE")
STRIDES_BACKEND = C.addressof(C.c_int.in_dll(lib, "CEED_STRIDES_BACKEND"))
_ERR_STORE = C.cast(lib.CeedErrorStore, C.c_void_p)
lib.CeedSetErrorHandler(None, _ERR_STORE)  # Python callers get exceptions, not abort()


def b2(rc):
    if rc:
        raise CeedError(f"b200 layer error {rc}: {lib.b200_last_error().decode()}")


def _ptr(a):
    """Raw address of a torch tensor / numpy array / int / None."""
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a.data_ptr()  # torch tensor


class _Obj:
    _destroy = None

    def __init__(self, ceed, handle):
        self.ceed, self.h = ceed, handle
        self._keep = []

    def _chk(self, rc):
        if rc:
            msg = C.c_char_p()
            lib.CeedGetErrorMessage(self.ceed.h if self.ceed is not None else None, C.byref(msg))
            raise CeedError(f"libceed_b200 error {rc}: {(msg.value or b'').decode()}")

    def destroy(self):
        if self.h is not None and self.h.value:
            getattr(lib, self._destroy)(C.byref(self.h))
            self.h = None


class Ceed(_Obj):
    """CeedInit(resource) -- /root/reference/elasticity.c:110"""
    _destroy = "CeedDestroy"

    def __init__(self, resource="/gpu/b200"):
        h = C.c_void_p()
        rc = lib.CeedInit(resource.encode(), C.byref(h))
        if rc or not h.value:
            msg = C.c_char_p()
            lib.CeedGetErrorMessage(None, C.byref(msg))
            raise CeedError(f"CeedInit({resource!r}) failed (rc={rc}): {(msg.value or b'').decode()}")
        super().__init__(None, h)
        self.ceed = self
        lib.CeedSetErrorHandler(h, _ERR_STORE)  # errors become Python exceptions instead of abort()

    def _chk(self, rc):
        if rc:
            msg = C.c_char_p()
            lib.CeedGetErrorMessage(self.h, C.byref(msg))
            raise CeedError(f"libceed_b200 error {rc}: {(msg.value or b'').decode()}")

    @property
    def resource(self):
        s = C.c_char_p()
        lib.CeedGetResource(self.h, C.byref(s))
        return s.value.decode()

    def preferred_memtype(self):
        m = C.c_int()
        lib.CeedGetPreferredMemType(self.h, C.byref(m))
        return m.value

    @property
    def is_deterministic(self):
        """CeedIsDeterministic: 1 for "/gpu/b200:deterministic" (ordered, atomic-free transposed restrictions)."""
        d = C.c_int()
        lib.CeedIsDeterministic(self.h, C.byref(d))
        return bool(d.value)

    def set_stream(self, cuda_stream_ptr):
        self._chk(lib.CeedB200SetStream(self.h, cuda_stream_ptr))

    def synchronize(self):
        self._chk(lib.CeedB200Synchronize(self.h))

    # factories
    def Vector(self, n):
        return Vector(self, n)

    def ElemRestriction(self, nelem, elemsize, ncomp, compstride, lsize, offsets):
        return ElemRestriction(self, nelem, elemsize, ncomp, compstride, lsize, offsets)

    def StridedElemRestriction(self, nelem, elemsize, ncomp, lsize, strides=None):
        return ElemRestriction(self, nelem, elemsize, ncomp, 0, lsize, None, strides=strides)

    def BasisTensorH1Lagrange(self, dim, ncomp, P, Q, qmode=GAUSS):
        return Basis(self, dim, ncomp, P, Q, qmode)

    def QFunction(self, vlength, source, f=None):
        return QFunction(self, vlength, source, f)

    def QFunctionIdentity(self, size, inmode, outmode):
        return QFunction(self, 1, None, identity=(size, inmode, outmode))

    def Operator(self, qf):
        return Operator(self, qf)


class Vector(_Obj):
    _destroy = "CeedVectorDestroy"

    def __init__(self, ceed, n):
        h = C.c_void_p()
        ceed._chk(lib.CeedVectorCreate(ceed.h, int(n), C.byref(h)))
        super().__init__(ceed, h)
        self.length = int(n)

    def set_array(self, array, mtype=None, cmode=USE_POINTER):
        """CeedVectorSetArray; array = torch tensor (device or host) or numpy array (host)."""
        if mtype is None:
            mtype = MEM_HOST if isinstance(array, np.ndarray) or not array.is_cuda else MEM_DEVICE
        if cmode != COPY_VALUES:
            self._keep = [array]
        self._chk(lib.CeedVectorSetArray(self.h, mtype, cmode, _ptr(array)))
        return self

    def take_array(self, mtype=MEM_DEVICE):
        """CeedVectorTakeArray(vec, mtype, NULL) -- matops.c:49-50"""
        self._chk(lib.CeedVectorTakeArray(self.h, mtype, None))
        self._keep = []

    def set_value(self, v):
        self._chk(lib.CeedVectorSetValue(self.h, float(v)))

    def to_numpy(self):
        p = C.c_void_p()
        self._chk(lib.CeedVectorGetArrayRead(self.h, MEM_HOST, C.byref(p)))
        out = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_double)), shape=(self.length,)).copy()
        self._chk(lib.CeedVectorRestoreArrayRead(self.h, C.byref(p)))
        return out

    def device_ptr(self, write=False):
        p = C.c_void_p()
        f = lib.CeedVectorGetArray if write else lib.CeedVectorGetArrayRead
        self._chk(f(self.h, MEM_DEVICE, C.byref(p)))
        return p.value

    def norm(self, ntype=NORM_2):
        r = C.c_double()
        self._chk(lib.CeedVectorNorm(self.h, ntype, C.byref(r)))
        return r.value

    def reciprocal(self):
        self._chk(lib.CeedVectorReciprocal(self.h))


class ElemRestriction(_Obj):
    _destroy = "CeedElemRestrictionDestroy"

    def __init__(self, ceed, nelem, elemsize, ncomp, compstride, lsize, offsets, strides=None):
        h = C.c_void_p()
        if offsets is not None:
            off = np.ascontiguousarray(offsets, dtype=np.int32)
            assert off.size == nelem * elemsize
            ceed._chk(lib.CeedElemRestrictionCreate(ceed.h, nelem, elemsize, ncomp, compstride, lsize, MEM_HOST,
                                                    COPY_VALUES, off.ctypes.data, C.byref(h)))
        else:
            if strides is None:
                sp = STRIDES_BACKEND
            else:
                sarr = (C.c_int * 3)(*strides)
                sp = C.addressof(sarr)
            ceed._chk(lib.CeedElemRestrictionCreateStrided(ceed.h, nelem, elemsize, ncomp, lsize, sp, C.byref(h)))
        super().__init__(ceed, h)
        self.nelem, self.elemsize, self.ncomp, self.lsize = nelem, elemsize, ncomp, lsize

    def create_vector(self):
        return Vector(self.ceed, self.lsize)

    def apply(self, u, ru, tmode=NOTRANSPOSE):
        self._chk(lib.CeedElemRestrictionApply(self.h, tmode, u.h, ru.h, REQUEST_IMMEDIATE))

    def get_multiplicity(self, mult):
        self._chk(lib.CeedElemRestrictionGetMultiplicity(self.h, mult.h))


class Basis(_Obj):
    _destroy = "CeedBasisDestroy"

    def __init__(self, ceed, dim, ncomp, P, Q, qmode):
        h = C.c_void_p()
        ceed._chk(lib.CeedBasisCreateTensorH1Lagrange(ceed.h, dim, ncomp, P, Q, qmode, C.byref(h)))
        super().__init__(ceed, h)
        self.dim, self.ncomp, self.P, self.Q = dim, ncomp, P, Q

    def _mat(self, getter, shape):
        p = C.c_void_p()
        getattr(lib, getter)(self.h, C.byref(p))
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_double)), shape=shape).copy()

    @property
    def interp1d(self):
        return self._mat("CeedBasisGetInterp1D", (self.Q, self.P))

    @property
    def grad1d(self):
        return self._mat("CeedBasisGetGrad1D", (self.Q, self.P))

    @property
    def qref1d(self):
        return self._mat("CeedBasisGetQRef", (self.Q,))

    @property
    def qweight1d(self):
        return self._mat("CeedBasisGetQWeights", (self.Q,))

    @property
    def num_qpts(self):
        n = C.c_int()
        lib.CeedBasisGetNumQuadraturePoints(self.h, C.byref(n))
        return n.value

    def apply(self, nelem, tmode, emode, u, v):
        self._chk(lib.CeedBasisApply(self.h, nelem, tmode, emode, u.h if u is not None else None, v.h))


class Physics(C.Structure):
    """Physics_private {nu, E} -- /root/reference/elasticity.h:30-37"""
    _fields_ = [("nu", C.c_double), ("E", C.c_double)]


class QFunction(_Obj):
    _destroy = "CeedQFunctionDestroy"

    def __init__(self, ceed, vlength, source, f=None, identity=None):
        h = C.c_void_p()
        if identity is not None:
            ceed._chk(lib.CeedQFunctionCreateIdentity(ceed.h, *identity, C.byref(h)))
        else:
            ceed._chk(lib.CeedQFunctionCreateInterior(ceed.h, vlength, f, source.encode(), C.byref(h)))
        super().__init__(ceed, h)

    def add_input(self, name, size, emode):
        self._chk(lib.CeedQFunctionAddInput(self.h, name.encode(), size, emode))

    def add_output(self, name, size, emode):
        self._chk(lib.CeedQFunctionAddOutput(self.h, name.encode(), size, emode))

    def set_context(self, ctx_struct, size=None):
        """The context stays a caller-owned host pointer (kept alive here)."""
        self._keep = [ctx_struct]
        self._chk(lib.CeedQFunctionSetContext(self.h, C.addressof(ctx_struct),
                                              C.sizeof(ctx_struct) if size is None else size))


class Operator(_Obj):
    _destroy = "CeedOperatorDestroy"

    def __init__(self, ceed, qf):
        h = C.c_void_p()
        ceed._chk(lib.CeedOperatorCreate(ceed.h, qf.h, QFUNCTION_NONE, QFUNCTION_NONE, C.byref(h)))
        super().__init__(ceed, h)
        self.qf = qf

    def set_field(self, name, r, b, v):
        rh = r.h if isinstance(r, _Obj) else r
        bh = b.h if isinstance(b, _Obj) else b
        vh = v.h if isinstance(v, _Obj) else v
        self._keep += [r, b, v]
        self._chk(lib.CeedOperatorSetField(self.h, name.encode(), rh, bh, vh))

    def apply(self, u, v):
        self._chk(lib.CeedOperatorApply(self.h, u.h, v.h, REQUEST_IMMEDIATE))

    def apply_add(self, u, v):
        self._chk(lib.CeedOperatorApplyAdd(self.h, u.h, v.h, REQUEST_IMMEDIATE))

    def apply_add_range(self, u, v, start, stop):
        self._chk(lib.CeedOperatorApplyAddRangeB200(self.h, u.h, v.h, int(start), int(stop)))

    def apply_partitioned(self, u, v, n_interface, halo_handle, mask_idx):
        """CeedOperatorApplyPartitionedB200: v = 0; interface elements; halo exchange overlapped with the interior
        elements; ordered sum; zero the entries mask_idx (int32 device tensor or None)."""
        self._chk(lib.CeedOperatorApplyPartitionedB200(
            self.h, u.h, v.h, int(n_interface), halo_handle,
            mask_idx.data_ptr() if mask_idx is not None and mask_idx.numel() else None,
            int(mask_idx.numel()) if mask_idx is not None else 0))

    def set_transfer_scaling(self, scale, inject=False):
        """CeedOperatorSetTransferScalingB200: fused transfer operators apply the fine-side inverse multiplicity
        themselves (matops.c:149,176); inject: the prolongation stores the interpolant instead of summing copies."""
        self._scale_keep = scale
        self._chk(lib.CeedOperatorSetTransferScalingB200(self.h, scale.h if scale is not None else None, int(bool(inject))))

    def linear_assemble_diagonal(self, assembled):
        self._chk(lib.CeedOperatorLinearAssembleDiagonal(self.h, assembled.h, REQUEST_IMMEDIATE))

    def linear_assemble_symbolic(self):
        """(rows, cols) int32 numpy arrays of the COO pattern (CeedOperatorLinearAssembleSymbolic)."""
        import numpy as np
        n = C.c_int()
        rows, cols = C.POINTER(_i)(), C.POINTER(_i)()
        self._chk(lib.CeedOperatorLinearAssembleSymbolic(self.h, C.byref(n), C.byref(rows), C.byref(cols)))
        r = np.ctypeslib.as_array(rows, shape=(max(n.value, 1),))[:n.value].copy()
        c = np.ctypeslib.as_array(cols, shape=(max(n.value, 1),))[:n.value].copy()
        libc = C.CDLL(None)
        libc.free.argtypes = [C.c_void_p]
        libc.free(rows)
        libc.free(cols)
        return r, c

    def linear_assemble(self, values):
        self._chk(lib.CeedOperatorLinearAssemble(self.h, values.h))

    @property
    def is_fused(self):
        f = C.c_int()
        self._chk(lib.CeedOperatorIsFusedB200(self.h, C.byref(f)))
        return bool(f.value)

    @property
    def is_jit_fused(self):
        """True if Apply runs the fused operator kernel generated around a JIT-compiled user QFunction (K12)"""
        f = C.c_int()
        self._chk(lib.CeedOperatorIsJitFusedB200(self.h, C.byref(f)))
        return bool(f.value)


def jit_compile(path, name, in_sizes, out_sizes):
    """The compile half of "/gpu/b200:jit" without a device: the QFunction `name` of the source file `path` (quoted
    includes inlined) with the given field sizes, compiled by NVRTC for sm_100a (cached per process).  Returns the
    handle; raises CeedError with the reason (unreadable file, NVRTC log)."""
    text, err = C.c_void_p(), C.create_string_buffer(1024)
    if lib.b200_jit_read_source(str(path).encode(), C.byref(text), err, len(err)):
        raise CeedError(err.value.decode())
    h = C.c_int(-1)
    try:
        rc = lib.b200_jit_compile(text, str(path).encode(), name.encode(), len(in_sizes), (C.c_int * 8)(*in_sizes),
                                  len(out_sizes), (C.c_int * 8)(*out_sizes), C.byref(h))
    finally:
        lib.b200_jit_free_source(text)
    b2(rc)
    return h.value


def jit_fused_compile(path, name, in_sizes, out_sizes, active_in, active_out, P, Q):
    """The compile half of K12 without a device: the fused operator kernel around QFunction `name` of `path` for the
    basis (P, Q), with field active_in / active_out as the active gradient and every other field passive (q-blocked).
    Returns the handle (cached per process, as jit_compile)."""
    text, err = C.c_void_p(), C.create_string_buffer(1024)
    if lib.b200_jit_read_source(str(path).encode(), C.byref(text), err, len(err)):
        raise CeedError(err.value.decode())
    h = C.c_int(-1)
    try:
        rc = lib.b200_jit_fused_compile(text, str(path).encode(), name.encode(), len(in_sizes),
                                        (C.c_int * 8)(*in_sizes), len(out_sizes), (C.c_int * 8)(*out_sizes),
                                        int(active_in), int(active_out), int(P), int(Q), C.byref(h))
    finally:
        lib.b200_jit_free_source(text)
    b2(rc)
    return h.value


def jit_assemble_compile(path, name, in_sizes, out_sizes, active_in, active_out, P, Q):
    """The compile half of K13 without a device: the element-matrix kernel of a trilinear level (P = 2) around
    QFunction `name` of `path`, fields as for jit_fused_compile.  Returns the handle (cached per process, as
    jit_compile)."""
    text, err = C.c_void_p(), C.create_string_buffer(1024)
    if lib.b200_jit_read_source(str(path).encode(), C.byref(text), err, len(err)):
        raise CeedError(err.value.decode())
    h = C.c_int(-1)
    try:
        rc = lib.b200_jit_assemble_compile(text, str(path).encode(), name.encode(), len(in_sizes),
                                           (C.c_int * 8)(*in_sizes), len(out_sizes), (C.c_int * 8)(*out_sizes),
                                           int(active_in), int(active_out), int(P), int(Q), C.byref(h))
    finally:
        lib.b200_jit_free_source(text)
    b2(rc)
    return h.value


def jit_program(handle):
    """Program text NVRTC compiled for a jit_compile handle (the user source with the generated kernel)."""
    p = lib.b200_jit_program(int(handle))
    return p.decode() if p is not None else None


def jit_compile_count():
    """NVRTC compilations run by this process (each distinct program is compiled once)."""
    return int(lib.b200_jit_compile_count())


def launch_count():
    return int(lib.CeedB200LaunchCount())


def launch_count_reset():
    lib.CeedB200LaunchCountReset()
