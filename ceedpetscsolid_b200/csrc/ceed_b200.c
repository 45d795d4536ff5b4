/* ceed_b200.c -- libCEED-compatible front-end + the "/gpu/b200" backend, in C99 over the
 * thin C-ABI CUDA layer (include/b200_kernels.h).
 *
 * What it mirrors (libCEED is not vendored in the reference; its call sites are):
 *   - the user API the reference calls (SURVEY.md App. A; /root/reference/src/setuplibceed.c,
 *     src/matops.c, src/misc.c, elasticity.c)
 *   - libCEED interface semantics: reference-counted objects, CeedOperatorApply = zero every
 *     output vector (active and passive) then ApplyAdd, fields matched by NAME between
 *     CeedQFunctionAdd{In,Out}put and CeedOperatorSetField, CEED_USE_POINTER borrows.
 *
 * Operator execution:
 *   FUSED     residual / Jacobian operators of the three material models -> one kernel
 *             (b200_apply_residual / b200_apply_jacobian); transfer operators -> b200_apply_transfer
 *   JIT_FUSED residual / Jacobian-shaped operators of a JIT-compiled user QFunction -> one generated kernel (K12,
 *             b200_jit_fused_apply), compiled at the operator's first apply; their diagonal -> K14
 *             (b200_jit_diag_apply), compiled at the operator's first diagonal
 *   GENERIC   everything else: restriction, basis and QFunction kernels chained on the device
 * There is no CPU fallback: a QFunction the backend does not recognise is an error, unless the resource carries
 * ":jit" -- then it is compiled from its source file with NVRTC (b200_jit.cu) and runs on K12 or the generic path.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "b200_kernels.h"
#include "ceed/ceed.h"

#define MAXF 8
#define B200_PIPE_MAXC 32
#define B200_PIPE_CHUNKS 16
#define B200_PIPE_MIN_ELEMS 8192 /* per chunk: enough CTAs to fill the GPU several times over */
#define CEED_B200_RESOURCE "/gpu/b200"
#define CEED_B200_ERRMSG 8192 /* room for an NVRTC log */

/* ------------------------------------------------------------------ objects */
typedef struct JCacheEntry {
  CeedVector qdata, gradu;
  int problem, nelem, Q;
  uint64_t vq, vg;
  double *d;
  struct JCacheEntry *next;
} JCacheEntry;

struct Ceed_private {
  char resource[128];
  int refcount;
  CeedErrorHandler eh;
  char errmsg[CEED_B200_ERRMSG];
  JCacheEntry *jcaches;
  /* "/gpu/b200:deterministic": transposed restrictions sum their E-vector in the serial /cpu/self order */
  int deterministic;
  /* "/gpu/b200:jit": QFunctions without a matching built-in body are compiled from their source file (op_setup) */
  int jit;
  double *det_evec;      /* device scratch E-vector shared by the fused kernels (stream-ordered reuse) */
  size_t det_evec_bytes;
};

struct CeedVector_private {
  Ceed ceed;
  int refcount;
  CeedInt length;
  double *h, *d;
  int h_owned, d_owned, h_valid, d_valid;
  uint64_t version;
};

struct CeedElemRestriction_private {
  Ceed ceed;
  int refcount;
  CeedInt nelem, elemsize, ncomp, compstride, lsize;
  int strided, backend_strides, layout_q, offsets_borrowed;
  CeedInt strides[3];
  int *d_offsets;
  int *d_tptr, *d_tidx;  /* deterministic mode: E-vector positions by offset value (CSR), built on first use */
  /* host-pipeline chunk tables (b200_apply_hostpipe), built on first use; pipe_n = -1: not worth it */
  int pipe_n, pipe_q;
  int pipe_end[B200_PIPE_MAXC];
  size_t pipe_in[B200_PIPE_MAXC], pipe_out[B200_PIPE_MAXC];
};

struct CeedBasis_private {
  Ceed ceed;
  int refcount;
  CeedInt dim, ncomp, P, Q;
  double *interp1d, *grad1d, *qref1d, *qweight1d;        /* host */
  double *d_interp1d, *d_grad1d, *d_qweight1d;           /* device, lazy */
};

typedef struct {
  char name[64];
  CeedInt size;
  CeedEvalMode emode;
} QFField;

struct CeedQFunction_private {
  Ceed ceed;
  int refcount;
  CeedInt vlength;
  CeedQFunctionUser f;
  char source[512], name[128];
  int qf_id;
  int nin, nout;
  QFField in[MAXF], out[MAXF];
  void *ctx;
  size_t ctxsize;
  int identity_size;
  int guard_done;  /* the caller's host function has been compared with the device body (qf_guard) */
  int jit_handle;  /* >= 0: runs the NVRTC-compiled kernel b200_jit_apply(jit_handle) instead of a built-in body */
  size_t jit_ctx_min; /* context bytes copied at least (what the built-in body of the same name reads) */
  char *jit_text;     /* the program text jit_handle was compiled from: K12 compiles it again around the fused kernel */
  char jit_path[512];
};

typedef struct {
  int set;
  CeedElemRestriction r;
  CeedBasis b;
  CeedVector v;
} OpField;

enum { OP_UNSET = 0, OP_GENERIC, OP_FUSED_RESIDUAL, OP_FUSED_JACOBIAN, OP_FUSED_TRANSFER, OP_JIT_FUSED };

struct CeedOperator_private {
  Ceed ceed;
  int refcount;
  CeedQFunction qf;
  OpField in[MAXF], out[MAXF];
  int kind, problem;
  int composite, nsubs;
  CeedOperator subs[MAXF];
  /* fused transfer operators: optional fine-side pointwise scaling (CeedOperatorSetTransferScalingB200) */
  CeedVector xfer_scale;
  int xfer_inject;
  /* ai / ao: the active input / output fields of a fused apply (0 / 0 for the built-in residual and Jacobian, whose
     QFunctions fix the field order; 0 for every other kind).  OP_JIT_FUSED: jit_fused = K12 program handle + 1 (0: not
     compiled yet); jit_assemble = K13 program handle + 1 (compiled at the first CeedOperatorLinearAssemble); jit_diag =
     K14 program handle + 1 (compiled at the first CeedOperatorLinearAssembleDiagonal) */
  int ai, ao, jit_fused, jit_assemble, jit_diag;
  /* generic-path work buffers (device), grown on demand */
  double *ebuf[2 * MAXF], *qbuf[2 * MAXF];
  size_t ebytes[2 * MAXF], qbytes[2 * MAXF];
};

/* ------------------------------------------------------------------ sentinels */
static struct CeedBasis_private basis_collocated_;
static struct CeedVector_private vector_active_, vector_none_;
static struct CeedElemRestriction_private rstr_none_;
static struct CeedQFunction_private qf_none_;
static CeedRequest req_immediate_, req_ordered_;
const CeedInt CEED_STRIDES_BACKEND[3] = {0, 0, 0};
const CeedBasis CEED_BASIS_COLLOCATED = &basis_collocated_;
const CeedVector CEED_VECTOR_ACTIVE = &vector_active_;
const CeedVector CEED_VECTOR_NONE = &vector_none_;
const CeedElemRestriction CEED_ELEMRESTRICTION_NONE = &rstr_none_;
const CeedQFunction CEED_QFUNCTION_NONE = &qf_none_;
CeedRequest *const CEED_REQUEST_IMMEDIATE = &req_immediate_;
CeedRequest *const CEED_REQUEST_ORDERED = &req_ordered_;
const char *const CeedMemTypes[] = {"host", "device", 0};
const char *const CeedEvalModes[] = {"none", "interpolation", "gradient", "", "divergence", "", "", "",
                                     "curl", "", "", "", "", "", "", "", "quadrature weights", 0};

/* ------------------------------------------------------------------ errors */
static char g_last_error[CEED_B200_ERRMSG];
static CeedErrorHandler g_default_eh = NULL; /* NULL = CeedErrorAbort (upstream default) */

int CeedErrorAbort(Ceed ceed, const char *file, int line, const char *func, int ecode, const char *format,
                   va_list *args) {
  (void)ceed;
  fprintf(stderr, "%s:%d in %s(): ", file, line, func);
  vfprintf(stderr, format, *args);
  fprintf(stderr, "\nAborted (libceed_b200, error %d)\n", ecode);
  abort();
  return ecode;
}
int CeedErrorReturn(Ceed ceed, const char *file, int line, const char *func, int ecode, const char *format,
                    va_list *args) {
  (void)ceed; (void)file; (void)line; (void)func; (void)format; (void)args;
  return ecode;
}
int CeedErrorStore(Ceed ceed, const char *file, int line, const char *func, int ecode, const char *format,
                   va_list *args) {
  char *dst = ceed ? ceed->errmsg : g_last_error;
  int n = snprintf(dst, CEED_B200_ERRMSG, "%s:%d in %s(): ", file, line, func);
  if (n < CEED_B200_ERRMSG) vsnprintf(dst + n, CEED_B200_ERRMSG - n, format, *args);
  if (ceed) memcpy(g_last_error, dst, CEED_B200_ERRMSG);
  return ecode;
}
static int CeedErrorImpl(Ceed ceed, const char *file, int line, const char *func, int ecode, const char *format, ...) {
  va_list args;
  va_start(args, format);
  CeedErrorHandler eh = ceed && ceed->eh ? ceed->eh : (g_default_eh ? g_default_eh : CeedErrorAbort);
  int rc = eh(ceed, file, line, func, ecode, format, &args);
  va_end(args);
  return rc;
}
#define CeedError(ceed, ecode, ...) CeedErrorImpl((ceed), __FILE__, __LINE__, __func__, (ecode), __VA_ARGS__)
#define CeedChk(ierr) do { int ierr_ = (ierr); if (ierr_) return ierr_; } while (0)
/* thin-layer call: turn a CUDA-layer failure into a Ceed error */
#define B2(ceed, call) do { int rc_ = (call); if (rc_) return CeedError((ceed), rc_, "%s: %s", #call, b200_last_error()); } while (0)

/* ceed == NULL sets the process-wide default used by CeedInit failures and new Ceed objects */
int CeedSetErrorHandler(Ceed ceed, CeedErrorHandler handler) {
  if (ceed) ceed->eh = handler;
  else g_default_eh = handler;
  return 0;
}
int CeedGetErrorMessage(Ceed ceed, const char **errmsg) { *errmsg = ceed ? ceed->errmsg : g_last_error; return 0; }
int CeedResetErrorMessage(Ceed ceed, const char **errmsg) {
  if (ceed) ceed->errmsg[0] = 0;
  g_last_error[0] = 0;
  if (errmsg) *errmsg = NULL;
  return 0;
}

/* ------------------------------------------------------------------ Ceed */
/* ":<word>" present as a whole qualifier of the resource */
static int has_qualifier(const char *resource, const char *word) {
  const size_t n = strlen(word);
  for (const char *p = strchr(resource, ':'); p; p = strchr(p + 1, ':'))
    if (!strncmp(p + 1, word, n) && (p[1 + n] == ':' || p[1 + n] == 0)) return 1;
  return 0;
}

int CeedInit(const char *resource, Ceed *ceed) {
  *ceed = NULL;
  if (!resource || strncmp(resource, CEED_B200_RESOURCE, strlen(CEED_B200_RESOURCE)))
    return CeedError(NULL, 1, "No suitable backend: %s (this library serves only %s; there is no CPU fallback)",
                     resource ? resource : "(null)", CEED_B200_RESOURCE);
  int ndev = 0;
  if (b200_device_count(&ndev) || ndev < 1)
    return CeedError(NULL, 2, "%s: no CUDA device visible (%s)", CEED_B200_RESOURCE, b200_last_error());
  /* optional "/gpu/b200:device_id=N" */
  const char *dv = strstr(resource, "device_id=");
  if (dv) {
    int id = atoi(dv + 10);
    if (id < 0 || id >= ndev) return CeedError(NULL, 2, "%s: device_id %d out of range", CEED_B200_RESOURCE, id);
    B2(NULL, b200_set_device(id));
  }
  Ceed c = (Ceed)calloc(1, sizeof *c);
  if (!c) return CeedError(NULL, 3, "out of memory");
  snprintf(c->resource, sizeof c->resource, "%s", resource);
  c->deterministic = strstr(resource, ":deterministic") != NULL;
  c->jit = has_qualifier(resource, "jit");
  c->refcount = 1;
  c->eh = g_default_eh ? g_default_eh : CeedErrorAbort;
  *ceed = c;
  return 0;
}

static void jcache_drop_for(Ceed ceed, CeedVector v) {
  JCacheEntry **p = &ceed->jcaches;
  while (*p) {
    if (!v || (*p)->qdata == v || (*p)->gradu == v) {
      JCacheEntry *dead = *p;
      *p = dead->next;
      b200_free(dead->d);
      free(dead);
    } else {
      p = &(*p)->next;
    }
  }
}

int CeedDestroy(Ceed *ceed) {
  if (!ceed || !*ceed) return 0;
  if (--(*ceed)->refcount > 0) { *ceed = NULL; return 0; }
  jcache_drop_for(*ceed, NULL);
  if ((*ceed)->det_evec) b200_free((*ceed)->det_evec);
  free(*ceed);
  *ceed = NULL;
  return 0;
}
int CeedGetResource(Ceed ceed, const char **resource) { *resource = ceed->resource; return 0; }
int CeedGetPreferredMemType(Ceed ceed, CeedMemType *type) { (void)ceed; *type = CEED_MEM_DEVICE; return 0; }
int CeedIsDeterministic(Ceed ceed, int *isDeterministic) { *isDeterministic = ceed->deterministic; return 0; }
int CeedB200SetStream(Ceed ceed, void *s) { B2(ceed, b200_set_stream(s)); return 0; }
int CeedB200Synchronize(Ceed ceed) { B2(ceed, b200_sync()); return 0; }
unsigned long long CeedB200LaunchCount(void) { return b200_launch_count(); }
void CeedB200LaunchCountReset(void) { b200_launch_count_reset(); }

/* ------------------------------------------------------------------ CeedVector */
int CeedVectorCreate(Ceed ceed, CeedInt len, CeedVector *vec) {
  if (len < 0) return CeedError(ceed, 1, "CeedVectorCreate: negative length %d", len);
  CeedVector v = (CeedVector)calloc(1, sizeof *v);
  if (!v) return CeedError(ceed, 3, "out of memory");
  v->ceed = ceed;
  ceed->refcount++;
  v->refcount = 1;
  v->length = len;
  *vec = v;
  return 0;
}

static size_t vbytes(CeedVector v) { return (size_t)v->length * sizeof(double); }

static int vec_alloc(CeedVector v, CeedMemType m) {
  if (m == CEED_MEM_HOST && !v->h) {
    v->h = (double *)malloc(vbytes(v) ? vbytes(v) : 8);
    if (!v->h) return CeedError(v->ceed, 3, "out of host memory (%zu bytes)", vbytes(v));
    v->h_owned = 1;
  } else if (m == CEED_MEM_DEVICE && !v->d) {
    B2(v->ceed, b200_malloc((void **)&v->d, vbytes(v)));
    v->d_owned = 1;
  }
  return 0;
}

static int vec_release(CeedVector v, CeedMemType m) {
  if (m == CEED_MEM_HOST) {
    if (v->h && v->h_owned) free(v->h);
    v->h = NULL; v->h_owned = 0; v->h_valid = 0;
  } else {
    if (v->d && v->d_owned) B2(v->ceed, b200_free(v->d));
    v->d = NULL; v->d_owned = 0; v->d_valid = 0;
  }
  return 0;
}

static int vec_sync(CeedVector v, CeedMemType m) {
  if (v->length == 0) { /* empty vectors (a rank without elements) are always "valid" */
    CeedChk(vec_alloc(v, m));
    if (m == CEED_MEM_HOST) v->h_valid = 1;
    else v->d_valid = 1;
    return 0;
  }
  if (m == CEED_MEM_HOST) {
    if (v->h_valid) return 0;
    if (!v->d_valid) return CeedError(v->ceed, 4, "CeedVector has no valid data (set it with CeedVectorSetArray/SetValue)");
    CeedChk(vec_alloc(v, CEED_MEM_HOST));
    B2(v->ceed, b200_memcpy_d2h(v->h, v->d, vbytes(v)));
    v->h_valid = 1;
  } else {
    if (v->d_valid) return 0;
    if (!v->h_valid) return CeedError(v->ceed, 4, "CeedVector has no valid data (set it with CeedVectorSetArray/SetValue)");
    CeedChk(vec_alloc(v, CEED_MEM_DEVICE));
    B2(v->ceed, b200_memcpy_h2d(v->d, v->h, vbytes(v)));
    v->d_valid = 1;
  }
  return 0;
}

/* backend-internal device access */
static int vec_dev_read(CeedVector v, const double **p) { CeedChk(vec_sync(v, CEED_MEM_DEVICE)); *p = v->d; return 0; }
static int vec_dev_write(CeedVector v, double **p) { /* contents undefined: caller overwrites everything */
  CeedChk(vec_alloc(v, CEED_MEM_DEVICE));
  v->d_valid = 1; v->h_valid = 0; v->version++;
  *p = v->d;
  return 0;
}
static int vec_dev_rw(CeedVector v, double **p) {
  CeedChk(vec_sync(v, CEED_MEM_DEVICE));
  v->h_valid = 0; v->version++;
  *p = v->d;
  return 0;
}

/* A host array borrowed with CEED_USE_POINTER is written in place by /cpu/self, and the reference relies on that:
 * ViewDiagnosticQuantities reads the borrowed array between CeedOperatorApply and CeedVectorTakeArray
 * (misc.c:258-268).  The public entry points that produce an output therefore bring a borrowed host array up to
 * date before they return; CeedVectorTakeArray then finds it current, so the MatMult path (matops.c:44-50) still
 * pays one device-to-host copy per product, not two. */
static int vec_write_through(CeedVector v) {
  if (!v || v == CEED_VECTOR_NONE || v == CEED_VECTOR_ACTIVE) return 0;
  if (v->h && !v->h_owned && !v->h_valid && v->d_valid) CeedChk(vec_sync(v, CEED_MEM_HOST));
  return 0;
}

int CeedVectorSetArray(CeedVector vec, CeedMemType mtype, CeedCopyMode cmode, CeedScalar *array) {
  Ceed ceed = vec->ceed;
  if (!array) return CeedError(ceed, 1, "CeedVectorSetArray: NULL array");
  if (mtype == CEED_MEM_HOST) {
    if (cmode == CEED_COPY_VALUES) {
      if (vec->h && !vec->h_owned) { vec->h = NULL; }
      CeedChk(vec_alloc(vec, CEED_MEM_HOST));
      memcpy(vec->h, array, vbytes(vec));
    } else {
      CeedChk(vec_release(vec, CEED_MEM_HOST));
      vec->h = array;
      vec->h_owned = cmode == CEED_OWN_POINTER;
    }
    vec->h_valid = 1; vec->d_valid = 0;
  } else {
    if (cmode == CEED_COPY_VALUES) {
      if (vec->d && !vec->d_owned) { vec->d = NULL; }
      CeedChk(vec_alloc(vec, CEED_MEM_DEVICE));
      B2(ceed, b200_memcpy_d2d(vec->d, array, vbytes(vec)));
    } else {
      CeedChk(vec_release(vec, CEED_MEM_DEVICE));
      vec->d = array;
      vec->d_owned = cmode == CEED_OWN_POINTER;
    }
    vec->d_valid = 1; vec->h_valid = 0;
  }
  vec->version++;
  return 0;
}

/* Ends a borrow (matops.c:49-50): the data is made current in `mtype` memory first, so a
 * host-borrowed output receives the device result here. */
int CeedVectorTakeArray(CeedVector vec, CeedMemType mtype, CeedScalar **array) {
  if (!vec->h_valid && !vec->d_valid) {
    if (array) *array = NULL;
    return 0;
  }
  CeedChk(vec_sync(vec, mtype));
  if (mtype == CEED_MEM_HOST) {
    if (array) *array = vec->h;
    else if (vec->h_owned) free(vec->h);
    vec->h = NULL; vec->h_owned = 0;
  } else {
    /* stream-ordered hand-back: work queued on the backend stream must be visible to the
       caller's next stream-ordered consumer (SURVEY 8(b)); both use the same stream. */
    if (array) *array = vec->d;
    else if (vec->d_owned) B2(vec->ceed, b200_free(vec->d));
    vec->d = NULL; vec->d_owned = 0;
  }
  vec->h_valid = vec->d_valid = 0;
  vec->version++;
  return 0;
}

int CeedVectorSetValue(CeedVector vec, CeedScalar value) {
  double *d;
  CeedChk(vec_dev_write(vec, &d));
  B2(vec->ceed, b200_vec_set(d, value, (size_t)vec->length));
  return 0;
}
int CeedVectorSyncArray(CeedVector vec, CeedMemType mtype) { return vec_sync(vec, mtype); }
int CeedVectorGetArray(CeedVector vec, CeedMemType mtype, CeedScalar **array) {
  CeedChk(vec_sync(vec, mtype));
  if (mtype == CEED_MEM_HOST) { vec->d_valid = 0; *array = vec->h; }
  else { vec->h_valid = 0; *array = vec->d; }
  vec->version++;
  return 0;
}
int CeedVectorGetArrayRead(CeedVector vec, CeedMemType mtype, const CeedScalar **array) {
  CeedChk(vec_sync(vec, mtype));
  *array = mtype == CEED_MEM_HOST ? vec->h : vec->d;
  return 0;
}
int CeedVectorRestoreArray(CeedVector vec, CeedScalar **array) { (void)vec; if (array) *array = NULL; return 0; }
int CeedVectorRestoreArrayRead(CeedVector vec, const CeedScalar **array) { (void)vec; if (array) *array = NULL; return 0; }
int CeedVectorNorm(CeedVector vec, CeedNormType type, CeedScalar *norm) {
  const double *d;
  CeedChk(vec_dev_read(vec, &d));
  B2(vec->ceed, b200_vec_norm_host(d, (size_t)vec->length, (int)type, norm));
  return 0;
}
int CeedVectorReciprocal(CeedVector vec) {
  double *d;
  CeedChk(vec_dev_rw(vec, &d));
  B2(vec->ceed, b200_vec_reciprocal(d, (size_t)vec->length));
  return 0;
}
int CeedVectorGetLength(CeedVector vec, CeedInt *length) { *length = vec->length; return 0; }
int CeedVectorDestroy(CeedVector *vec) {
  if (!vec || !*vec) return 0;
  CeedVector v = *vec;
  *vec = NULL;
  if (v == CEED_VECTOR_ACTIVE || v == CEED_VECTOR_NONE) return 0;
  if (--v->refcount > 0) return 0;
  jcache_drop_for(v->ceed, v);
  vec_release(v, CEED_MEM_HOST);
  vec_release(v, CEED_MEM_DEVICE);
  Ceed c = v->ceed;
  free(v);
  return CeedDestroy(&c);
}

/* ------------------------------------------------------------------ CeedElemRestriction */
int CeedElemRestrictionCreate(Ceed ceed, CeedInt nelem, CeedInt elemsize, CeedInt ncomp, CeedInt compstride,
                              CeedInt lsize, CeedMemType mtype, CeedCopyMode cmode, const CeedInt *offsets,
                              CeedElemRestriction *rstr) {
  if (!offsets) return CeedError(ceed, 1, "CeedElemRestrictionCreate: NULL offsets");
  CeedElemRestriction r = (CeedElemRestriction)calloc(1, sizeof *r);
  if (!r) return CeedError(ceed, 3, "out of memory");
  r->ceed = ceed; ceed->refcount++; r->refcount = 1;
  r->nelem = nelem; r->elemsize = elemsize; r->ncomp = ncomp; r->compstride = compstride; r->lsize = lsize;
  const size_t n = (size_t)nelem * elemsize;
  if (mtype == CEED_MEM_HOST) {
    for (size_t i = 0; i < n; i++) {
      const long long hi = (long long)offsets[i] + (long long)(ncomp - 1) * compstride;
      if (offsets[i] < 0 || hi >= lsize) {
        free(r); ceed->refcount--;
        return CeedError(ceed, 1, "CeedElemRestrictionCreate: offset %d at position %zu out of range [0,%d)", offsets[i], i, lsize);
      }
    }
    B2(ceed, b200_malloc((void **)&r->d_offsets, n * sizeof(int)));
    B2(ceed, b200_memcpy_h2d(r->d_offsets, offsets, n * sizeof(int)));
    B2(ceed, b200_sync());  /* caller may free its array right away (setuplibceed.c:235-237) */
    if (cmode == CEED_OWN_POINTER) free((void *)offsets);
  } else {
    if (cmode == CEED_COPY_VALUES) {
      B2(ceed, b200_malloc((void **)&r->d_offsets, n * sizeof(int)));
      B2(ceed, b200_memcpy_d2d(r->d_offsets, offsets, n * sizeof(int)));
    } else {
      r->d_offsets = (int *)offsets; /* USE/OWN device pointer: kept, never freed here unless owned */
      r->offsets_borrowed = cmode == CEED_USE_POINTER;
    }
  }
  *rstr = r;
  return 0;
}

int CeedElemRestrictionCreateStrided(Ceed ceed, CeedInt nelem, CeedInt elemsize, CeedInt ncomp, CeedInt lsize,
                                     const CeedInt strides[3], CeedElemRestriction *rstr) {
  CeedElemRestriction r = (CeedElemRestriction)calloc(1, sizeof *r);
  if (!r) return CeedError(ceed, 3, "out of memory");
  r->ceed = ceed; ceed->refcount++; r->refcount = 1;
  r->nelem = nelem; r->elemsize = elemsize; r->ncomp = ncomp; r->compstride = 0; r->lsize = lsize;
  r->strided = 1;
  if (strides == CEED_STRIDES_BACKEND || (strides[0] == 0 && strides[1] == 0 && strides[2] == 0)) {
    r->backend_strides = 1;
    r->layout_q = b200_strided_layout_q(elemsize);  /* q-blocked when elemsize = Q^3 */
    r->strides[0] = 1; r->strides[1] = elemsize; r->strides[2] = elemsize * ncomp; /* plain layout otherwise */
  } else {
    memcpy(r->strides, strides, 3 * sizeof(CeedInt));
  }
  if ((long long)nelem * elemsize * ncomp > lsize) {
    free(r); ceed->refcount--;
    return CeedError(ceed, 1, "CeedElemRestrictionCreateStrided: lsize %d too small for %d x %d x %d", lsize, nelem, elemsize, ncomp);
  }
  *rstr = r;
  return 0;
}

int CeedElemRestrictionCreateVector(CeedElemRestriction rstr, CeedVector *lvec, CeedVector *evec) {
  if (lvec) CeedChk(CeedVectorCreate(rstr->ceed, rstr->lsize, lvec));
  if (evec) CeedChk(CeedVectorCreate(rstr->ceed, rstr->nelem * rstr->elemsize * rstr->ncomp, evec));
  return 0;
}

/* deterministic mode: CSR of the E-vector positions p = e*elemsize + n by offset value, ascending p */
static int rstr_transpose_map(CeedElemRestriction r) {
  Ceed ceed = r->ceed;
  if (r->d_tptr) return 0;
  const size_t n = (size_t)r->nelem * r->elemsize;
  int *off = (int *)malloc((n ? n : 1) * sizeof(int)), *tptr = (int *)malloc(((size_t)r->lsize + 1) * sizeof(int));
  int *tidx = (int *)malloc((n ? n : 1) * sizeof(int));
  if (!off || !tptr || !tidx) { free(off); free(tptr); free(tidx); return CeedError(ceed, 3, "out of memory"); }
  int rc = b200_memcpy_d2h(off, r->d_offsets, n * sizeof(int));
  if (!rc) rc = b200_transpose_map_build(r->lsize, n, off, tptr, tidx);
  if (!rc) rc = b200_malloc((void **)&r->d_tptr, ((size_t)r->lsize + 1) * sizeof(int));
  if (!rc) rc = b200_malloc((void **)&r->d_tidx, (n ? n : 1) * sizeof(int));
  if (!rc) rc = b200_memcpy_h2d(r->d_tptr, tptr, ((size_t)r->lsize + 1) * sizeof(int));
  if (!rc) rc = b200_memcpy_h2d(r->d_tidx, tidx, n * sizeof(int));
  if (!rc) rc = b200_sync();
  free(off); free(tptr); free(tidx);
  if (rc) return CeedError(ceed, rc, "deterministic restriction map: %s", b200_last_error());
  return 0;
}

/* L += E^T E-vector in the serial (element, node) order; layout as b200_transpose_gather_add */
static int rstr_ordered_add(CeedElemRestriction r, int layout, const double *evec, double *L) {
  CeedChk(rstr_transpose_map(r));
  B2(r->ceed, b200_transpose_gather_add(r->lsize, r->d_tptr, r->d_tidx, r->elemsize, r->ncomp, r->compstride, layout, evec, L));
  return 0;
}

/* deterministic mode: the Ceed's scratch E-vector, grown to a transposed restriction through r, which the caller sums
   into the L-vector with rstr_ordered_add; NULL otherwise (the kernels add with atomics) */
static int det_evec(Ceed ceed, CeedElemRestriction r, double **evec) {
  const size_t bytes = (size_t)r->nelem * r->elemsize * r->ncomp * sizeof(double);
  *evec = NULL;
  if (!ceed->deterministic) return 0;
  if (ceed->det_evec_bytes < bytes) {
    if (ceed->det_evec) { B2(ceed, b200_sync()); B2(ceed, b200_free(ceed->det_evec)); ceed->det_evec = NULL; ceed->det_evec_bytes = 0; }
    B2(ceed, b200_malloc((void **)&ceed->det_evec, bytes));
    ceed->det_evec_bytes = bytes;
  }
  *evec = ceed->det_evec;
  return 0;
}

static int rstr_apply_raw(CeedElemRestriction r, int transpose, const double *in, double *out) {
  if (transpose && !r->strided && r->ceed->deterministic) return rstr_ordered_add(r, 0, in, out);
  if (r->strided == 1)
    B2(r->ceed, b200_restrict_strided(transpose, r->nelem, r->elemsize, r->ncomp, r->backend_strides ? r->layout_q : 0,
                                      r->strides[0], r->strides[1], r->strides[2], in, out));
  else
    B2(r->ceed, b200_restrict_offsets(transpose, r->nelem, r->elemsize, r->ncomp, r->compstride, r->d_offsets, in, out));
  return 0;
}

/* NOTRANSPOSE: ru = E u (overwrites);  TRANSPOSE: ru += E^T u  (upstream semantics) */
int CeedElemRestrictionApply(CeedElemRestriction rstr, CeedTransposeMode tmode, CeedVector u, CeedVector ru,
                             CeedRequest *request) {
  (void)request;
  const double *in;
  double *out;
  CeedChk(vec_dev_read(u, &in));
  if (tmode == CEED_NOTRANSPOSE) CeedChk(vec_dev_write(ru, &out));
  else CeedChk(vec_dev_rw(ru, &out));
  return rstr_apply_raw(rstr, tmode == CEED_TRANSPOSE, in, out);
}

/* misc.c:117-123: transpose-apply of an E-vector of ones into a zeroed L-vector */
int CeedElemRestrictionGetMultiplicity(CeedElemRestriction rstr, CeedVector mult) {
  Ceed ceed = rstr->ceed;
  const size_t n = (size_t)rstr->nelem * rstr->elemsize * rstr->ncomp;
  double *ones, *m;
  B2(ceed, b200_malloc((void **)&ones, n * sizeof(double)));
  B2(ceed, b200_vec_set(ones, 1.0, n));
  CeedChk(vec_dev_write(mult, &m));
  B2(ceed, b200_vec_set(m, 0.0, (size_t)mult->length));
  CeedChk(rstr_apply_raw(rstr, 1, ones, m));
  B2(ceed, b200_sync());
  B2(ceed, b200_free(ones));
  return vec_write_through(mult);
}
int CeedElemRestrictionGetNumElements(CeedElemRestriction r, CeedInt *n) { *n = r->nelem; return 0; }
int CeedElemRestrictionGetElementSize(CeedElemRestriction r, CeedInt *n) { *n = r->elemsize; return 0; }
int CeedElemRestrictionGetLVectorSize(CeedElemRestriction r, CeedInt *n) { *n = r->lsize; return 0; }
int CeedElemRestrictionGetNumComponents(CeedElemRestriction r, CeedInt *n) { *n = r->ncomp; return 0; }
int CeedElemRestrictionDestroy(CeedElemRestriction *rstr) {
  if (!rstr || !*rstr) return 0;
  CeedElemRestriction r = *rstr;
  *rstr = NULL;
  if (r == CEED_ELEMRESTRICTION_NONE) return 0;
  if (--r->refcount > 0) return 0;
  if (r->d_offsets && !r->offsets_borrowed) b200_free(r->d_offsets);
  if (r->d_tptr) b200_free(r->d_tptr);
  if (r->d_tidx) b200_free(r->d_tidx);
  Ceed c = r->ceed;
  free(r);
  return CeedDestroy(&c);
}

/* ------------------------------------------------------------------ CeedBasis */
static void legendre_pair(int n, double x, double *Pn, double *Pnm1) {
  double a = 1.0, b = x;
  if (n == 0) { *Pn = 1.0; *Pnm1 = 0.0; return; }
  for (int j = 2; j <= n; j++) { const double c = ((2 * j - 1) * x * b - (j - 1) * a) / j; a = b; b = c; }
  *Pn = b; *Pnm1 = a;
}

int CeedGaussQuadrature(CeedInt Q, CeedScalar *x, CeedScalar *w) {
  const double pi = 4.0 * atan(1.0);
  for (int i = 0; i <= Q / 2; i++) {
    double xi = cos(pi * (2 * i + 1) / (2.0 * Q)), p, pm, dp = 1;
    for (int it = 0; it < 100; it++) {
      legendre_pair(Q, xi, &p, &pm);
      dp = (xi * p - pm) * Q / (xi * xi - 1.0);
      const double step = p / dp;
      xi -= step;
      if (fabs(step) < 1e-16 || fabs(p) < 1e-15) break;
    }
    legendre_pair(Q, xi, &p, &pm);
    dp = (xi * p - pm) * Q / (xi * xi - 1.0);
    w[i] = w[Q - 1 - i] = 2.0 / ((1.0 - xi * xi) * dp * dp);
    x[i] = -xi; x[Q - 1 - i] = xi;
  }
  return 0;
}

int CeedLobattoQuadrature(CeedInt Q, CeedScalar *x, CeedScalar *w) {
  const double pi = 4.0 * atan(1.0);
  const int n = Q - 1;
  if (Q < 2) return 1;
  x[0] = -1.0; x[Q - 1] = 1.0;
  if (w) w[0] = w[Q - 1] = 2.0 / (Q * (double)n);
  for (int i = 1; i <= n / 2; i++) {
    double xi = cos(pi * i / n), p, pm;
    for (int it = 0; it < 100; it++) {
      legendre_pair(n, xi, &p, &pm);
      const double dp = (xi * p - pm) * n / (xi * xi - 1.0);
      const double d2p = (2 * xi * dp - n * (n + 1.0) * p) / (1.0 - xi * xi);
      const double step = dp / d2p;
      xi -= step;
      if (fabs(step) < 1e-16) break;
    }
    legendre_pair(n, xi, &p, &pm);
    if (w) w[i] = w[Q - 1 - i] = 2.0 / (Q * (double)n * p * p);
    x[i] = -xi; x[Q - 1 - i] = xi;
  }
  return 0;
}

int CeedBasisCreateTensorH1(Ceed ceed, CeedInt dim, CeedInt ncomp, CeedInt P, CeedInt Q, const CeedScalar *interp1d,
                            const CeedScalar *grad1d, const CeedScalar *qref1d, const CeedScalar *qweight1d,
                            CeedBasis *basis) {
  if (dim != 3) return CeedError(ceed, 1, "%s supports dim = 3 tensor bases (got %d)", CEED_B200_RESOURCE, dim);
  if (P < 1 || Q < 1) return CeedError(ceed, 1, "CeedBasisCreateTensorH1: P, Q must be positive");
  CeedBasis b = (CeedBasis)calloc(1, sizeof *b);
  if (!b) return CeedError(ceed, 3, "out of memory");
  b->ceed = ceed; ceed->refcount++; b->refcount = 1;
  b->dim = dim; b->ncomp = ncomp; b->P = P; b->Q = Q;
  b->interp1d = (double *)malloc(sizeof(double) * Q * P);
  b->grad1d = (double *)malloc(sizeof(double) * Q * P);
  b->qref1d = (double *)malloc(sizeof(double) * Q);
  b->qweight1d = (double *)malloc(sizeof(double) * Q);
  memcpy(b->interp1d, interp1d, sizeof(double) * Q * P);
  memcpy(b->grad1d, grad1d, sizeof(double) * Q * P);
  memcpy(b->qref1d, qref1d, sizeof(double) * Q);
  memcpy(b->qweight1d, qweight1d, sizeof(double) * Q);
  *basis = b;
  return 0;
}

/* GLL nodes; Gauss or GLL quadrature; Lagrange interp/grad by Fornberg's recurrence */
int CeedBasisCreateTensorH1Lagrange(Ceed ceed, CeedInt dim, CeedInt ncomp, CeedInt P, CeedInt Q, CeedQuadMode qmode,
                                    CeedBasis *basis) {
  if (P < 2 || Q < 1 || P > 16 || Q > 16) return CeedError(ceed, 1, "CeedBasisCreateTensorH1Lagrange: need 2 <= P <= 16, 1 <= Q <= 16");
  double nodes[16], qref[16], qw[16], B[256], D[256];
  CeedLobattoQuadrature(P, nodes, NULL);
  if (qmode == CEED_GAUSS) CeedGaussQuadrature(Q, qref, qw);
  else if (Q >= 2) CeedLobattoQuadrature(Q, qref, qw);
  else return CeedError(ceed, 1, "Gauss-Lobatto needs Q >= 2");
  for (int i = 0; i < Q; i++) {
    double *b = B + i * P, *d = D + i * P;
    for (int j = 0; j < P; j++) b[j] = d[j] = 0.0;
    double c1 = 1.0, c3 = nodes[0] - qref[i];
    b[0] = 1.0;
    for (int j = 1; j < P; j++) {
      double c2 = 1.0;
      const double c4 = c3;
      c3 = nodes[j] - qref[i];
      for (int k = 0; k < j; k++) {
        const double dx = nodes[j] - nodes[k];
        c2 *= dx;
        if (k == j - 1) {
          d[j] = c1 * (b[k] - c4 * d[k]) / c2;
          b[j] = -c1 * c4 * b[k] / c2;
        }
        d[k] = (c3 * d[k] - b[k]) / dx;
        b[k] = c3 * b[k] / dx;
      }
      c1 = c2;
    }
  }
  /* at a point that is one of the nodes the Lagrange basis is exactly a unit vector; the recurrence can round it
   * (1 + 2^-52 at the end point of the Pc = 4 -> Pf = 5 Gauss-Lobatto interpolation), and then two elements sharing a
   * fine node of the p-multigrid prolongation interpolate different values there */
  for (int i = 0; i < Q; i++)
    for (int j = 0; j < P; j++)
      if (qref[i] == nodes[j])
        for (int k = 0; k < P; k++) B[i * P + k] = k == j ? 1.0 : 0.0;
  return CeedBasisCreateTensorH1(ceed, dim, ncomp, P, Q, B, D, qref, qw, basis);
}

static int basis_device(CeedBasis b) {
  if (b->d_interp1d) return 0;
  const size_t n = sizeof(double) * b->Q * b->P;
  B2(b->ceed, b200_malloc((void **)&b->d_interp1d, n));
  B2(b->ceed, b200_malloc((void **)&b->d_grad1d, n));
  B2(b->ceed, b200_malloc((void **)&b->d_qweight1d, sizeof(double) * b->Q));
  B2(b->ceed, b200_memcpy_h2d(b->d_interp1d, b->interp1d, n));
  B2(b->ceed, b200_memcpy_h2d(b->d_grad1d, b->grad1d, n));
  B2(b->ceed, b200_memcpy_h2d(b->d_qweight1d, b->qweight1d, sizeof(double) * b->Q));
  B2(b->ceed, b200_sync());
  return 0;
}

static int emode_to_b200(CeedEvalMode e) { return e == CEED_EVAL_INTERP ? 1 : e == CEED_EVAL_GRAD ? 2 : e == CEED_EVAL_WEIGHT ? 4 : 0; }

static int basis_apply_raw(CeedBasis b, CeedInt nelem, int transpose, CeedEvalMode emode, const double *u, double *v) {
  const int em = emode_to_b200(emode);
  if (!em) return CeedError(b->ceed, 1, "CeedBasisApply: eval mode %d not supported by %s", (int)emode, CEED_B200_RESOURCE);
  CeedChk(basis_device(b));
  B2(b->ceed, b200_basis_apply(nelem, b->ncomp, b->P, b->Q, b->d_interp1d, b->d_grad1d, b->d_qweight1d, transpose, em, u, v));
  return 0;
}

int CeedBasisApply(CeedBasis basis, CeedInt nelem, CeedTransposeMode tmode, CeedEvalMode emode, CeedVector u, CeedVector v) {
  const double *in = NULL;
  double *out;
  if (emode != CEED_EVAL_WEIGHT) CeedChk(vec_dev_read(u, &in));
  CeedChk(vec_dev_write(v, &out));
  return basis_apply_raw(basis, nelem, tmode == CEED_TRANSPOSE, emode, in, out);
}
int CeedBasisGetNumNodes(CeedBasis b, CeedInt *P) { *P = b->P * b->P * b->P; return 0; }
int CeedBasisGetNumQuadraturePoints(CeedBasis b, CeedInt *Q) { *Q = b->Q * b->Q * b->Q; return 0; }
int CeedBasisGetInterp1D(CeedBasis b, const CeedScalar **p) { *p = b->interp1d; return 0; }
int CeedBasisGetGrad1D(CeedBasis b, const CeedScalar **p) { *p = b->grad1d; return 0; }
int CeedBasisGetQRef(CeedBasis b, const CeedScalar **p) { *p = b->qref1d; return 0; }
int CeedBasisGetQWeights(CeedBasis b, const CeedScalar **p) { *p = b->qweight1d; return 0; }
int CeedBasisDestroy(CeedBasis *basis) {
  if (!basis || !*basis) return 0;
  CeedBasis b = *basis;
  *basis = NULL;
  if (b == CEED_BASIS_COLLOCATED) return 0;
  if (--b->refcount > 0) return 0;
  free(b->interp1d); free(b->grad1d); free(b->qref1d); free(b->qweight1d);
  b200_free(b->d_interp1d); b200_free(b->d_grad1d); b200_free(b->d_qweight1d);
  Ceed c = b->ceed;
  free(b);
  return CeedDestroy(&c);
}

/* ------------------------------------------------------------------ CeedQFunction */
static int qf_lookup(const char *name) {
  static const struct { const char *n; int id; } table[] = {
      {"SetupGeo", B200_QF_SETUPGEO},     {"LinElasF", B200_QF_LINELAS_F},   {"LinElasdF", B200_QF_LINELAS_DF},
      {"HyperSSF", B200_QF_HYPERSS_F},    {"HyperSSdF", B200_QF_HYPERSS_DF}, {"HyperFSF", B200_QF_HYPERFS_F},
      {"HyperFSdF", B200_QF_HYPERFS_DF},  {"Identity", B200_QF_IDENTITY},    {"SetupConstantForce", B200_QF_CONST_FORCE},
      {"SetupMMSForce", B200_QF_MMS_FORCE}, {"MMSTrueSoln", B200_QF_MMS_TRUE},
      {"LinElasEnergy", B200_QF_LINELAS_ENERGY}, {"HyperSSEnergy", B200_QF_HYPERSS_ENERGY},
      {"HyperFSEnergy", B200_QF_HYPERFS_ENERGY}, {"LinElasDiagnostic", B200_QF_LINELAS_DIAG},
      {"HyperSSDiagnostic", B200_QF_HYPERSS_DIAG}, {"HyperFSDiagnostic", B200_QF_HYPERFS_DIAG}, {NULL, 0}};
  for (int i = 0; table[i].n; i++)
    if (!strcmp(table[i].n, name)) return table[i].id;
  return B200_QF_NONE;
}

int CeedQFunctionCreateInterior(Ceed ceed, CeedInt vlength, CeedQFunctionUser f, const char *source, CeedQFunction *qf) {
  CeedQFunction q = (CeedQFunction)calloc(1, sizeof *q);
  if (!q) return CeedError(ceed, 3, "out of memory");
  q->ceed = ceed; ceed->refcount++; q->refcount = 1;
  q->vlength = vlength; q->f = f;
  snprintf(q->source, sizeof q->source, "%s", source ? source : "");
  const char *colon = strrchr(q->source, ':');
  snprintf(q->name, sizeof q->name, "%s", colon ? colon + 1 : q->source);
  q->qf_id = qf_lookup(q->name); /* unknown names are reported when an operator tries to run them */
  q->jit_handle = -1;
  *qf = q;
  return 0;
}

int CeedQFunctionCreateIdentity(Ceed ceed, CeedInt size, CeedEvalMode inmode, CeedEvalMode outmode, CeedQFunction *qf) {
  CeedChk(CeedQFunctionCreateInterior(ceed, 1, NULL, "gallery:Identity", qf));
  (*qf)->identity_size = size;
  CeedChk(CeedQFunctionAddInput(*qf, "input", size, inmode));
  CeedChk(CeedQFunctionAddOutput(*qf, "output", size, outmode));
  return 0;
}

static int qf_add(CeedQFunction qf, QFField *arr, int *n, const char *name, CeedInt size, CeedEvalMode emode) {
  if (*n >= MAXF) return CeedError(qf->ceed, 1, "too many QFunction fields (max %d)", MAXF);
  snprintf(arr[*n].name, sizeof arr[*n].name, "%s", name);
  arr[*n].size = size; arr[*n].emode = emode;
  (*n)++;
  return 0;
}
int CeedQFunctionAddInput(CeedQFunction qf, const char *fieldname, CeedInt size, CeedEvalMode emode) {
  return qf_add(qf, qf->in, &qf->nin, fieldname, size, emode);
}
int CeedQFunctionAddOutput(CeedQFunction qf, const char *fieldname, CeedInt size, CeedEvalMode emode) {
  if (emode == CEED_EVAL_WEIGHT) return CeedError(qf->ceed, 1, "CEED_EVAL_WEIGHT is not a valid output mode");
  return qf_add(qf, qf->out, &qf->nout, fieldname, size, emode);
}
/* The context stays a caller-owned HOST pointer that is re-read at every apply: the reference
 * passes sizeof(pointer) instead of sizeof(struct) at setuplibceed.c:826, and swaps the
 * context around the diagonal assembly (matops.c:215-217,231-232). */
int CeedQFunctionSetContext(CeedQFunction qf, void *ctx, size_t ctxsize) { qf->ctx = ctx; qf->ctxsize = ctxsize; return 0; }
int CeedQFunctionDestroy(CeedQFunction *qf) {
  if (!qf || !*qf) return 0;
  CeedQFunction q = *qf;
  *qf = NULL;
  if (q == CEED_QFUNCTION_NONE) return 0;
  if (--q->refcount > 0) return 0;
  Ceed c = q->ceed;
  b200_jit_free_source(q->jit_text);
  free(q);
  return CeedDestroy(&c);
}

/* ------------------------------------------------------------------ CeedOperator */
int CeedOperatorCreate(Ceed ceed, CeedQFunction qf, CeedQFunction dqf, CeedQFunction dqfT, CeedOperator *op) {
  (void)dqf; (void)dqfT;
  if (!qf || qf == CEED_QFUNCTION_NONE) return CeedError(ceed, 1, "CeedOperatorCreate: a QFunction is required");
  CeedOperator o = (CeedOperator)calloc(1, sizeof *o);
  if (!o) return CeedError(ceed, 3, "out of memory");
  o->ceed = ceed; ceed->refcount++; o->refcount = 1;
  o->qf = qf; qf->refcount++;
  *op = o;
  return 0;
}
int CeedCompositeOperatorCreate(Ceed ceed, CeedOperator *op) {
  CeedOperator o = (CeedOperator)calloc(1, sizeof *o);
  if (!o) return CeedError(ceed, 3, "out of memory");
  o->ceed = ceed; ceed->refcount++; o->refcount = 1; o->composite = 1;
  *op = o;
  return 0;
}
int CeedCompositeOperatorAddSub(CeedOperator comp, CeedOperator sub) {
  if (!comp->composite) return CeedError(comp->ceed, 1, "CeedCompositeOperatorAddSub: not a composite operator");
  if (comp->nsubs >= MAXF) return CeedError(comp->ceed, 1, "too many sub-operators");
  comp->subs[comp->nsubs++] = sub;
  sub->refcount++;
  return 0;
}

int CeedOperatorSetField(CeedOperator op, const char *fieldname, CeedElemRestriction r, CeedBasis b, CeedVector v) {
  if (op->composite) return CeedError(op->ceed, 1, "CeedOperatorSetField on a composite operator");
  OpField *f = NULL;
  for (int i = 0; i < op->qf->nin && !f; i++)
    if (!strcmp(op->qf->in[i].name, fieldname)) f = &op->in[i];
  for (int i = 0; i < op->qf->nout && !f; i++)
    if (!strcmp(op->qf->out[i].name, fieldname)) f = &op->out[i];
  if (!f) return CeedError(op->ceed, 1, "CeedOperatorSetField: QFunction %s has no field \"%s\"", op->qf->name, fieldname);
  if (f->set) return CeedError(op->ceed, 1, "CeedOperatorSetField: field \"%s\" already set", fieldname);
  f->set = 1; f->r = r; f->b = b; f->v = v;
  if (r && r != CEED_ELEMRESTRICTION_NONE) r->refcount++;
  if (b && b != CEED_BASIS_COLLOCATED) b->refcount++;
  if (v && v != CEED_VECTOR_ACTIVE && v != CEED_VECTOR_NONE) v->refcount++;
  op->kind = OP_UNSET;
  return 0;
}

static int is_tensor3(CeedBasis b) { return b && b != CEED_BASIS_COLLOCATED && b->dim == 3; }
static int is_qstrided(CeedElemRestriction r, int ncomp, int Q) {
  return r && r != CEED_ELEMRESTRICTION_NONE && r->strided == 1 && r->backend_strides && r->layout_q == Q && r->ncomp == ncomp;
}
static int is_passive(CeedVector v) { return v && v != CEED_VECTOR_ACTIVE && v != CEED_VECTOR_NONE; }

/* classify once all fields are set */
/* The reference hands over a host function pointer AND a source locator (setuplibceed.c:370-372, 518-520, 818-820);
 * this backend dispatches on the NAME in the locator to a hand-written device body and never executes the pointer on
 * the data path.  A locally edited qfunctions header would then silently run the stock body -- so, once per QFunction,
 * the caller's own function is run on the host on a few known points and compared with the device body evaluated on
 * the host (b200_qfunction_apply_host: the same __host__ __device__ code).  A mismatch is a loud error.  Covers the
 * hot-path QFunctions (SetupGeo, residual F and Jacobian dF of the three models); skipped when no host pointer was
 * given (bindings without one) or CEED_B200_SKIP_QF_GUARD is set. */
static int qf_guard(CeedQFunction qf, int *differs) {
  Ceed ceed = qf->ceed;
  if (qf->guard_done || !qf->f || getenv("CEED_B200_SKIP_QF_GUARD")) return 0;
  const int id = qf->qf_id;
  if (id < B200_QF_SETUPGEO || id > B200_QF_HYPERFS_DF) return 0;
  enum { NQ = 3 };
  double hctx[2] = {0.3, 1.0};
  if (id != B200_QF_SETUPGEO) {
    if (!qf->ctx) return 0;  /* context not set yet: checked at the next set-up */
    memcpy(hctx, qf->ctx, sizeof hctx);
  }
  /* known points: a mildly distorted geometry (J near diag(0.5, 0.4, 0.6)) and displacement gradients of a few % */
  static const double Jref[NQ][9] = {{0.50, 0.02, -0.01, 0.03, 0.40, 0.02, -0.02, 0.01, 0.60},
                                     {0.45, -0.03, 0.02, 0.01, 0.42, -0.02, 0.03, 0.02, 0.55},
                                     {0.52, 0.01, 0.03, -0.02, 0.38, 0.01, 0.01, -0.03, 0.62}};
  static const double wref[NQ] = {0.31, 0.17, 0.26};
  static const double gref[NQ][9] = {{0.031, -0.012, 0.007, 0.015, -0.024, 0.011, -0.008, 0.019, 0.027},
                                     {-0.022, 0.017, 0.013, -0.009, 0.033, -0.016, 0.021, -0.005, -0.014},
                                     {0.012, 0.026, -0.019, 0.023, 0.008, 0.017, -0.011, -0.028, 0.035}};
  double qdata[10 * NQ], in_buf[MAXF][10 * NQ], out_user[MAXF][10 * NQ], out_dev[MAXF][10 * NQ];
  { /* qdata from the backend's own SetupGeo body */
    double dx[9 * NQ], w[NQ];
    for (int q = 0; q < NQ; q++) {
      for (int k = 0; k < 9; k++) dx[k * NQ + q] = Jref[q][k];
      w[q] = wref[q];
    }
    const double *gin[2] = {dx, w};
    double *gout[1] = {qdata};
    B2(ceed, b200_qfunction_apply_host(B200_QF_SETUPGEO, NULL, 0, 0, 1, NQ, 2, gin, 1, gout));
  }
  const double *in[MAXF];
  double *outu[MAXF], *outd[MAXF];
  for (int i = 0; i < qf->nin; i++) {
    const QFField *f = &qf->in[i];
    if (f->size > 10) return 0;
    for (int q = 0; q < NQ; q++)
      for (int k = 0; k < f->size; k++) {
        double v;
        if (f->size == 10) v = qdata[k * NQ + q];
        else if (f->emode == CEED_EVAL_WEIGHT || f->size == 1) v = wref[q];
        else if (id == B200_QF_SETUPGEO) v = Jref[q][k % 9];
        else if (f->emode == CEED_EVAL_GRAD) v = gref[(q + 1) % NQ][k % 9] * 1.3;   /* du / deltadu */
        else v = gref[q][k % 9];                                                  /* stored gradu */
        in_buf[i][k * NQ + q] = v;
      }
    in[i] = in_buf[i];
  }
  for (int i = 0; i < qf->nout; i++) {
    if (qf->out[i].size > 10) return 0;
    memset(out_user[i], 0, sizeof out_user[i]);
    memset(out_dev[i], 0, sizeof out_dev[i]);
    outu[i] = out_user[i];
    outd[i] = out_dev[i];
  }
  const int rc_user = qf->f(qf->ctx, NQ, in, outu);
  if (rc_user) return CeedError(ceed, 1, "QFunction %s (%s): the caller's function returned %d on the known-answer points", qf->name, qf->source, rc_user);
  B2(ceed, b200_qfunction_apply_host(id, hctx, id == B200_QF_SETUPGEO ? 0 : 2, 0, 1, NQ, qf->nin, in, qf->nout, outd));
  for (int i = 0; i < qf->nout; i++) {
    double scale = 0, diff = 0;
    for (int k = 0; k < qf->out[i].size * NQ; k++) {
      if (fabs(out_user[i][k]) > scale) scale = fabs(out_user[i][k]);
      if (fabs(out_user[i][k] - out_dev[i][k]) > diff) diff = fabs(out_user[i][k] - out_dev[i][k]);
    }
    if (!(diff <= 1e-10 * (scale > 1e-300 ? scale : 1e-300))) {
      if (differs) { /* "/gpu/b200:jit": op_setup compiles the caller's source instead */
        *differs = 1;
        return 0;
      }
      return CeedError(ceed, 1,
                       "%s: the QFunction at %s does not compute what this backend's device body for \"%s\" computes "
                       "(output \"%s\": max difference %.3e at scale %.3e on the known-answer points).  The backend runs its "
                       "own hand-written body for the names it recognises and would silently ignore a modified source; "
                       "there is no CPU fallback (the \":jit\" resource qualifier compiles the source instead).",
                       CEED_B200_RESOURCE, qf->source, qf->name, qf->out[i].name, diff, scale);
    }
  }
  qf->guard_done = 1;
  return 0;
}

/* "/gpu/b200:jit": compile the QFunction from the file of its "<file>:<Name>" locator (b200_jit.cu) */
static int qf_jit_compile(CeedQFunction qf, int guard_differs) {
  Ceed ceed = qf->ceed;
  const char *why = guard_differs ? " (the QFunction guard found that the caller's function differs from this backend's "
                                    "built-in body for this name, so it is compiled from its source)" : "";
  const char *colon = strrchr(qf->source, ':');
  if (!colon || colon == qf->source)
    return CeedError(ceed, 1, "%s: QFunction \"%s\": locator \"%s\" names no source file (\"<file>:<Name>\")%s",
                     CEED_B200_RESOURCE, qf->name, qf->source, why);
  char path[sizeof qf->source], err[1024];
  snprintf(path, sizeof path, "%.*s", (int)(colon - qf->source), qf->source);
  char *text = NULL;
  if (b200_jit_read_source(path, &text, err, sizeof err))
    return CeedError(ceed, 1, "%s: QFunction \"%s\": %s%s", CEED_B200_RESOURCE, qf->name, err, why);
  int in_sizes[MAXF], out_sizes[MAXF], h = -1;
  for (int i = 0; i < qf->nin; i++) in_sizes[i] = qf->in[i].size;
  for (int i = 0; i < qf->nout; i++) out_sizes[i] = qf->out[i].size;
  const int rc = b200_jit_compile(text, path, qf->name, qf->nin, in_sizes, qf->nout, out_sizes, &h);
  if (rc) {
    b200_jit_free_source(text);
    return CeedError(ceed, rc, "%s: QFunction \"%s\" from %s: %s%s", CEED_B200_RESOURCE, qf->name, path, b200_last_error(), why);
  }
  qf->jit_handle = h;
  b200_jit_free_source(qf->jit_text);
  qf->jit_text = text;
  snprintf(qf->jit_path, sizeof qf->jit_path, "%s", path);
  /* the reference declares the Physics context with sizeof(pointer) (setuplibceed.c:826); the built-in bodies read
     {nu, E} whatever ctxsize says, so a guard-routed material model gets at least those 16 bytes too */
  qf->jit_ctx_min = guard_differs && qf->qf_id != B200_QF_SETUPGEO ? sizeof(b200_physics) : 0;
  return 0;
}

/* the active fields of the fused kernels: input ai an active EVAL_GRAD of 9 on a 3-component offsets restriction
 * (compstride 1, P^3 nodes) with a tensor basis whose (P, Q) has a fused layout, output ao an active EVAL_GRAD of 9 on
 * the same restriction and the same basis matrices */
static int fused_active_shape(CeedOperator op, int ai, int ao) {
  CeedQFunction qf = op->qf;
  OpField *u = &op->in[ai], *vv = &op->out[ao];
  if (!(qf->in[ai].emode == CEED_EVAL_GRAD && qf->in[ai].size == 9 && u->v == CEED_VECTOR_ACTIVE && is_tensor3(u->b) &&
        u->b->ncomp == 3 && u->r && u->r != CEED_ELEMRESTRICTION_NONE && u->r->strided == 0 && u->r->ncomp == 3 &&
        u->r->compstride == 1 && u->r->elemsize == u->b->P * u->b->P * u->b->P && b200_fused_supported(u->b->P, u->b->Q)))
    return 0;
  const int Q = u->b->Q;
  return qf->out[ao].emode == CEED_EVAL_GRAD && qf->out[ao].size == 9 && vv->v == CEED_VECTOR_ACTIVE && vv->r == u->r &&
         (vv->b == u->b || (is_tensor3(vv->b) && vv->b->P == u->b->P && vv->b->Q == Q &&
                            !memcmp(vv->b->interp1d, u->b->interp1d, sizeof(double) * Q * u->b->P) &&
                            !memcmp(vv->b->grad1d, u->b->grad1d, sizeof(double) * Q * u->b->P)));
}

/* K12 (OP_JIT_FUSED): one active input and one active output of the fused active shape, and every other field
 * EVAL_NONE on a passive vector with a q-blocked restriction of the same nelem */
static int jit_fused_eligible(CeedOperator op) {
  CeedQFunction qf = op->qf;
  int ai = -1, ao = -1;
  for (int i = 0; i < qf->nin; i++)
    if (op->in[i].v == CEED_VECTOR_ACTIVE) { if (ai >= 0) return 0; ai = i; }
  for (int i = 0; i < qf->nout; i++)
    if (op->out[i].v == CEED_VECTOR_ACTIVE) { if (ao >= 0) return 0; ao = i; }
  if (ai < 0 || ao < 0 || !fused_active_shape(op, ai, ao)) return 0;
  OpField *u = &op->in[ai];
  const int Q = u->b->Q;
  for (int i = 0; i < qf->nin + qf->nout; i++) {
    if (i == ai || i == qf->nin + ao) continue;
    const QFField *qff = i < qf->nin ? &qf->in[i] : &qf->out[i - qf->nin];
    OpField *f = i < qf->nin ? &op->in[i] : &op->out[i - qf->nin];
    if (!(qff->emode == CEED_EVAL_NONE && is_passive(f->v) && is_qstrided(f->r, qff->size, Q) &&
          f->r->nelem == u->r->nelem && (size_t)f->v->length >= (size_t)f->r->nelem * qff->size * Q * Q * Q))
      return 0;
  }
  op->ai = ai;
  op->ao = ao;
  return 1;
}

static int op_setup(CeedOperator op) {
  CeedQFunction qf = op->qf;
  for (int i = 0; i < qf->nin; i++)
    if (!op->in[i].set) return CeedError(op->ceed, 1, "operator field \"%s\" of QFunction %s not set", qf->in[i].name, qf->name);
  for (int i = 0; i < qf->nout; i++)
    if (!op->out[i].set) return CeedError(op->ceed, 1, "operator field \"%s\" of QFunction %s not set", qf->out[i].name, qf->name);
  /* "/gpu/b200:jit": an unknown name, or a recognised one whose caller function the guard finds different, is compiled
     from its source and runs on the generic path; gallery:Identity and a passing (or impossible) guard keep the
     built-in body */
  if (op->ceed->jit && qf->jit_handle < 0 && qf->qf_id != B200_QF_IDENTITY) {
    int differs = 0;
    if (qf->qf_id != B200_QF_NONE) CeedChk(qf_guard(qf, &differs));
    if (qf->qf_id == B200_QF_NONE || differs) CeedChk(qf_jit_compile(qf, differs));
  }
  op->ai = op->ao = 0;
  op->jit_fused = 0;
  op->jit_assemble = 0;
  op->jit_diag = 0;
  if (qf->jit_handle >= 0) {
    op->kind = qf->jit_text && jit_fused_eligible(op) ? OP_JIT_FUSED : OP_GENERIC;
    return 0;
  }
  if (qf->qf_id == B200_QF_NONE)
    return CeedError(op->ceed, 1,
                     "%s: QFunction \"%s\" (%s) is not one this backend has a device body for; there is no CPU fallback "
                     "(the \":jit\" resource qualifier compiles it from its source)",
                     CEED_B200_RESOURCE, qf->name, qf->source);
  CeedChk(qf_guard(qf, NULL));
  op->kind = OP_GENERIC;
  const int id = qf->qf_id;
  const int is_res = id == B200_QF_LINELAS_F || id == B200_QF_HYPERSS_F || id == B200_QF_HYPERFS_F;
  const int is_jac = id == B200_QF_LINELAS_DF || id == B200_QF_HYPERSS_DF || id == B200_QF_HYPERFS_DF;
  if (is_res || is_jac) {
    const int prob = (id == B200_QF_LINELAS_F || id == B200_QF_LINELAS_DF) ? B200_PROB_LINELAS
                     : (id == B200_QF_HYPERSS_F || id == B200_QF_HYPERSS_DF) ? B200_PROB_HYPERSS : B200_PROB_HYPERFS;
    const int has_gradu = prob != B200_PROB_LINELAS;
    const int nin = is_jac && has_gradu ? 3 : 2, nout = is_res && has_gradu ? 2 : 1;
    int ok = qf->nin == nin && qf->nout == nout && fused_active_shape(op, 0, 0);
    if (ok) {
      OpField *u = &op->in[0], *qd = &op->in[1];
      const int Q = u->b->Q;
      ok = qf->in[1].emode == CEED_EVAL_NONE && qf->in[1].size == 10 && is_qstrided(qd->r, 10, Q) && is_passive(qd->v) &&
           qd->r->nelem == u->r->nelem;
      if (ok && has_gradu) {
        OpField *g = is_jac ? &op->in[2] : &op->out[1];
        const QFField *gf = is_jac ? &qf->in[2] : &qf->out[1];
        ok = gf->emode == CEED_EVAL_NONE && gf->size == 9 && is_qstrided(g->r, 9, Q) && is_passive(g->v) &&
             g->r->nelem == u->r->nelem;
      }
    }
    if (ok) {
      op->kind = is_res ? OP_FUSED_RESIDUAL : OP_FUSED_JACOBIAN;
      op->problem = prob;
    }
  } else if (id == B200_QF_IDENTITY && qf->nin == 1 && qf->nout == 1 && qf->identity_size == 3) {
    /* p-MG transfer (setuplibceed.c:847-863): prolong = coarse INTERP(basisCtoF) -> fine NONE;
       restrict = fine NONE -> coarse INTERP(basisCtoF)^T */
    OpField *i0 = &op->in[0], *o0 = &op->out[0];
    const int prolong = qf->in[0].emode == CEED_EVAL_INTERP && qf->out[0].emode == CEED_EVAL_NONE;
    const int restr = qf->in[0].emode == CEED_EVAL_NONE && qf->out[0].emode == CEED_EVAL_INTERP;
    if ((prolong || restr) && i0->v == CEED_VECTOR_ACTIVE && o0->v == CEED_VECTOR_ACTIVE) {
      OpField *c = prolong ? i0 : o0, *f = prolong ? o0 : i0;
      static const int pairs[][2] = {{2, 3}, {3, 4}, {4, 5}, {3, 5}, {2, 4}, {2, 5}};
      if (is_tensor3(c->b) && c->r && f->r && c->r != CEED_ELEMRESTRICTION_NONE && f->r != CEED_ELEMRESTRICTION_NONE &&
          c->r->strided == 0 && f->r->strided == 0 && c->r->ncomp == 3 && f->r->ncomp == 3 && c->r->compstride == 1 &&
          f->r->compstride == 1 && c->r->nelem == f->r->nelem && c->b->ncomp == 3 &&
          c->r->elemsize == c->b->P * c->b->P * c->b->P && f->r->elemsize == c->b->Q * c->b->Q * c->b->Q)
        for (size_t k = 0; k < sizeof pairs / sizeof pairs[0]; k++)
          if (pairs[k][0] == c->b->P && pairs[k][1] == c->b->Q) op->kind = OP_FUSED_TRANSFER;
    }
  }
  return 0;
}

/* the operators whose apply runs on the fused kernels, element range by element range: the built-in residual and
   Jacobian, and K12 */
static int op_fused_apply(CeedOperator op) {
  return op->kind == OP_FUSED_JACOBIAN || op->kind == OP_FUSED_RESIDUAL || op->kind == OP_JIT_FUSED;
}

/* the operators whose diagonal and p = 1 assembly run on fused kernels: the built-in Jacobians (the linear-elastic
   residual is its own Jacobian), and the JIT operators of K12 */
static int op_fused_jacobian(CeedOperator op) {
  return op->kind == OP_FUSED_JACOBIAN || op->kind == OP_JIT_FUSED ||
         (op->kind == OP_FUSED_RESIDUAL && op->problem == B200_PROB_LINELAS);
}

int CeedOperatorIsFusedB200(CeedOperator op, int *isFused) {
  if (op->composite) { *isFused = 0; return 0; }
  if (op->kind == OP_UNSET) CeedChk(op_setup(op));
  *isFused = op->kind != OP_GENERIC && op->kind != OP_JIT_FUSED;
  return 0;
}

int CeedOperatorIsJitFusedB200(CeedOperator op, int *isJitFused) {
  if (op->composite) { *isJitFused = 0; return 0; }
  if (op->kind == OP_UNSET) CeedChk(op_setup(op));
  *isJitFused = op->kind == OP_JIT_FUSED;
  return 0;
}

static int qf_physics(CeedQFunction qf, b200_physics *phys) {
  if (!qf->ctx) return CeedError(qf->ceed, 1, "QFunction %s needs a Physics context (CeedQFunctionSetContext)", qf->name);
  memcpy(phys, qf->ctx, sizeof *phys); /* {nu, E}: read through the host pointer, whatever ctxsize says */
  return 0;
}

/* Jacobian cache for (qdata[, gradu]) -- rebuilt when either vector changed */
static int jcache_get(CeedOperator op, const double **jc) {
  Ceed ceed = op->ceed;
  const int prob = op->problem;
  CeedVector qd = op->in[1].v, gu = prob == B200_PROB_LINELAS ? NULL : op->in[2].v;
  const int nelem = op->in[0].r->nelem, Q = op->in[0].b->Q;
  JCacheEntry *e = ceed->jcaches;
  while (e && !(e->qdata == qd && e->gradu == gu && e->problem == prob)) e = e->next;
  if (!e) {
    e = (JCacheEntry *)calloc(1, sizeof *e);
    if (!e) return CeedError(ceed, 3, "out of memory");
    e->qdata = qd; e->gradu = gu; e->problem = prob; e->nelem = nelem; e->Q = Q;
    e->vq = e->vg = (uint64_t)-1;
    const size_t bytes = sizeof(double) * (size_t)b200_jcache_ncomp(prob) * nelem * Q * Q * Q;
    int rc = b200_malloc((void **)&e->d, bytes);
    if (rc) { free(e); return CeedError(ceed, rc, "Jacobian cache allocation (%zu bytes): %s", bytes, b200_last_error()); }
    e->next = ceed->jcaches;
    ceed->jcaches = e;
  }
  if (e->vq != qd->version || (gu && e->vg != gu->version)) {
    const double *q, *g = NULL;
    CeedChk(vec_dev_read(qd, &q));
    if (gu) CeedChk(vec_dev_read(gu, &g));
    B2(ceed, b200_jcache_build(prob, nelem, Q, q, g, e->d));
    e->vq = qd->version;
    if (gu) e->vg = gu->version;
  }
  *jc = e->d;
  return 0;
}

static int grow(Ceed ceed, double **buf, size_t *have, size_t need) {
  if (*have >= need) return 0;
  if (*buf) { B2(ceed, b200_sync()); B2(ceed, b200_free(*buf)); *buf = NULL; *have = 0; }
  B2(ceed, b200_malloc((void **)buf, need));
  *have = need;
  return 0;
}

/* element / quadrature-point counts of a generic operator */
static int op_counts(CeedOperator op, CeedInt *nelem_out, CeedInt *nq_out) {
  Ceed ceed = op->ceed;
  CeedQFunction qf = op->qf;
  CeedInt nelem = 0, nq = 0;
  for (int i = 0; i < qf->nin + qf->nout; i++) {
    OpField *f = i < qf->nin ? &op->in[i] : &op->out[i - qf->nin];
    const CeedEvalMode em = i < qf->nin ? qf->in[i].emode : qf->out[i - qf->nin].emode;
    if (f->r && f->r != CEED_ELEMRESTRICTION_NONE) {
      if (nelem && nelem != f->r->nelem) return CeedError(ceed, 1, "operator fields disagree on the number of elements");
      nelem = f->r->nelem;
    }
    if (em != CEED_EVAL_NONE && is_tensor3(f->b)) nq = f->b->Q * f->b->Q * f->b->Q;
  }
  if (!nq)
    for (int i = 0; i < qf->nin && !nq; i++)
      if (op->in[i].r && op->in[i].r != CEED_ELEMRESTRICTION_NONE) nq = op->in[i].r->elemsize;
  if (!nelem || !nq) return CeedError(ceed, 1, "operator %s: cannot determine element / quadrature counts", qf->name);
  *nelem_out = nelem;
  *nq_out = nq;
  return 0;
}

/* Q-vector of input field i (restriction + basis); `in` feeds active fields.  With
 * skip_active the active fields are left to the caller (diagonal assembly). */
static int op_input_qvec(CeedOperator op, int i, CeedVector in, CeedInt nelem, CeedInt nq, int skip_active,
                         const double **q) {
  Ceed ceed = op->ceed;
  CeedQFunction qf = op->qf;
  OpField *f = &op->in[i];
  const CeedEvalMode em = qf->in[i].emode;
  const size_t qsz = sizeof(double) * (size_t)nelem * qf->in[i].size * nq;
  *q = NULL;
  if (em == CEED_EVAL_WEIGHT) {
    if (!is_tensor3(f->b)) return CeedError(ceed, 1, "field \"%s\": CEED_EVAL_WEIGHT needs a basis", qf->in[i].name);
    CeedChk(grow(ceed, &op->qbuf[i], &op->qbytes[i], qsz));
    CeedChk(basis_apply_raw(f->b, nelem, 0, CEED_EVAL_WEIGHT, NULL, op->qbuf[i]));
    *q = op->qbuf[i];
    return 0;
  }
  if (f->v == CEED_VECTOR_ACTIVE && skip_active) return 0;
  CeedVector src = f->v == CEED_VECTOR_ACTIVE ? in : f->v;
  if (!src || src == CEED_VECTOR_NONE) return CeedError(ceed, 1, "field \"%s\" has no input vector", qf->in[i].name);
  if (!f->r || f->r == CEED_ELEMRESTRICTION_NONE) return CeedError(ceed, 1, "field \"%s\" needs an element restriction", qf->in[i].name);
  const double *l;
  CeedChk(vec_dev_read(src, &l));
  const size_t esz = sizeof(double) * (size_t)nelem * f->r->ncomp * f->r->elemsize;
  CeedChk(grow(ceed, &op->ebuf[i], &op->ebytes[i], esz));
  CeedChk(rstr_apply_raw(f->r, 0, l, op->ebuf[i]));
  if (em == CEED_EVAL_NONE) {
    if (f->r->elemsize != nq || f->r->ncomp != qf->in[i].size)
      return CeedError(ceed, 1, "field \"%s\": CEED_EVAL_NONE size mismatch", qf->in[i].name);
    *q = op->ebuf[i];
  } else {
    if (!is_tensor3(f->b)) return CeedError(ceed, 1, "field \"%s\": eval mode needs a tensor basis", qf->in[i].name);
    if (qf->in[i].size != f->b->ncomp * (em == CEED_EVAL_GRAD ? 3 : 1))
      return CeedError(ceed, 1, "field \"%s\": QFunction size %d does not match basis", qf->in[i].name, qf->in[i].size);
    CeedChk(grow(ceed, &op->qbuf[i], &op->qbytes[i], qsz));
    CeedChk(basis_apply_raw(f->b, nelem, 0, em, op->ebuf[i], op->qbuf[i]));
    *q = op->qbuf[i];
  }
  return 0;
}

/* context bytes of a JIT-compiled QFunction: copied from the caller's host pointer at every apply, as for the built-in
   bodies */
static int jit_ctx_bytes(CeedQFunction qf, size_t *bytes) {
  Ceed ceed = qf->ceed;
  *bytes = qf->ctxsize > qf->jit_ctx_min ? qf->ctxsize : qf->jit_ctx_min;
  if (*bytes > B200_JIT_MAX_CTX)
    return CeedError(ceed, 1, "%s: QFunction %s has a context of %zu bytes; a JIT-compiled QFunction takes at most %d",
                     CEED_B200_RESOURCE, qf->name, *bytes, B200_JIT_MAX_CTX);
  if (*bytes && !qf->ctx) return CeedError(ceed, 1, "QFunction %s needs a context (CeedQFunctionSetContext)", qf->name);
  return 0;
}

static int op_run_qfunction(CeedOperator op, CeedInt nelem, CeedInt nq, const double **qin, double **qout) {
  Ceed ceed = op->ceed;
  CeedQFunction qf = op->qf;
  for (int i = 0; i < qf->nout; i++) {
    const size_t qsz = sizeof(double) * (size_t)nelem * qf->out[i].size * nq;
    CeedChk(grow(ceed, &op->qbuf[MAXF + i], &op->qbytes[MAXF + i], qsz));
    qout[i] = op->qbuf[MAXF + i];
  }
  if (qf->jit_handle >= 0) {
    size_t bytes;
    CeedChk(jit_ctx_bytes(qf, &bytes));
    B2(ceed, b200_jit_apply(qf->jit_handle, qf->ctx, bytes, nelem, nq, qf->nin, qin, qf->nout, qout));
    return 0;
  }
  /* context: read through the caller's host pointer at apply time, whatever ctxsize says
     (Physics {nu, E}: 2 doubles; constant forcing vector: 3 doubles, declared as sizeof(double),
     setuplibceed.c:566-567) */
  double hctx[4] = {0, 0, 0, 0};
  int nctx = 0;
  const int id = qf->qf_id;
  if (id == B200_QF_CONST_FORCE) nctx = 3;
  else if (id != B200_QF_SETUPGEO && id != B200_QF_IDENTITY && id != B200_QF_MMS_TRUE) nctx = 2;
  if (nctx) {
    if (!qf->ctx) return CeedError(ceed, 1, "QFunction %s needs a context (CeedQFunctionSetContext)", qf->name);
    memcpy(hctx, qf->ctx, sizeof(double) * nctx);
  }
  B2(ceed, b200_qfunction_apply(id, hctx, nctx, qf->identity_size, nelem, nq, qf->nin, qin, qf->nout, qout));
  return 0;
}

static int op_apply_generic(CeedOperator op, CeedVector in, CeedVector out) {
  Ceed ceed = op->ceed;
  CeedQFunction qf = op->qf;
  CeedInt nelem = 0, nq = 0;
  CeedChk(op_counts(op, &nelem, &nq));
  const double *qin[MAXF];
  double *qout[MAXF];
  for (int i = 0; i < qf->nin; i++) CeedChk(op_input_qvec(op, i, in, nelem, nq, 0, &qin[i]));
  CeedChk(op_run_qfunction(op, nelem, nq, qin, qout));
  for (int i = 0; i < qf->nout; i++) {
    OpField *f = &op->out[i];
    const CeedEvalMode em = qf->out[i].emode;
    CeedVector dst = f->v == CEED_VECTOR_ACTIVE ? out : f->v;
    if (!dst || dst == CEED_VECTOR_NONE) return CeedError(ceed, 1, "field \"%s\" has no output vector", qf->out[i].name);
    if (!f->r || f->r == CEED_ELEMRESTRICTION_NONE) return CeedError(ceed, 1, "field \"%s\" needs an element restriction", qf->out[i].name);
    double *l;
    CeedChk(vec_dev_rw(dst, &l));
    const double *e = qout[i];
    if (em != CEED_EVAL_NONE) {
      if (!is_tensor3(f->b)) return CeedError(ceed, 1, "field \"%s\": eval mode needs a tensor basis", qf->out[i].name);
      const size_t esz = sizeof(double) * (size_t)nelem * f->r->ncomp * f->r->elemsize;
      CeedChk(grow(ceed, &op->ebuf[MAXF + i], &op->ebytes[MAXF + i], esz));
      CeedChk(basis_apply_raw(f->b, nelem, 1, em, qout[i], op->ebuf[MAXF + i]));
      e = op->ebuf[MAXF + i];
    } else if (f->r->elemsize != nq || f->r->ncomp != qf->out[i].size) {
      return CeedError(ceed, 1, "field \"%s\": CEED_EVAL_NONE size mismatch", qf->out[i].name);
    }
    CeedChk(rstr_apply_raw(f->r, 1, e, l));
  }
  return 0;
}

/* Generic CeedOperatorLinearAssembleAddDiagonal (App. B.5) for operators of the Jacobian shape:
 * one active GRAD input and one active GRAD output on the same restriction and basis.  Nine
 * unit-input QFunction passes, each folded into the element diagonal on the device. */
static int op_diagonal_generic(CeedOperator op, CeedVector assembled) {
  Ceed ceed = op->ceed;
  CeedQFunction qf = op->qf;
  int ia = -1, oa = -1;
  for (int i = 0; i < qf->nin; i++)
    if (op->in[i].v == CEED_VECTOR_ACTIVE) ia = ia < 0 ? i : -2;
  for (int i = 0; i < qf->nout; i++)
    if (op->out[i].v == CEED_VECTOR_ACTIVE) oa = oa < 0 ? i : -2;
  if (ia < 0 || oa < 0 || qf->nout != 1 || qf->in[ia].emode != CEED_EVAL_GRAD || qf->out[oa].emode != CEED_EVAL_GRAD ||
      qf->in[ia].size != 9 || qf->out[oa].size != 9 || !is_tensor3(op->in[ia].b) || op->in[ia].r != op->out[oa].r ||
      !op->in[ia].r || op->in[ia].r == CEED_ELEMRESTRICTION_NONE)
    return CeedError(ceed, 1, "%s: CeedOperatorLinearAssembleDiagonal supports operators with one active 3-component "
                              "GRAD input and output on the same restriction (QFunction %s does not qualify)",
                     CEED_B200_RESOURCE, qf->name);
  CeedInt nelem = 0, nq = 0;
  CeedChk(op_counts(op, &nelem, &nq));
  CeedBasis b = op->in[ia].b;
  CeedElemRestriction r = op->in[ia].r;
  CeedChk(basis_device(b));
  const double *qin[MAXF];
  double *qout[MAXF];
  for (int i = 0; i < qf->nin; i++) CeedChk(op_input_qvec(op, i, NULL, nelem, nq, 1, &qin[i]));
  const size_t usz = sizeof(double) * (size_t)nelem * 9 * nq, esz = sizeof(double) * (size_t)nelem * 3 * r->elemsize;
  CeedChk(grow(ceed, &op->qbuf[ia], &op->qbytes[ia], usz));
  CeedChk(grow(ceed, &op->ebuf[MAXF + oa], &op->ebytes[MAXF + oa], esz));
  double *unit = op->qbuf[ia], *ediag = op->ebuf[MAXF + oa];
  qin[ia] = unit;
  B2(ceed, b200_memset(ediag, 0, esz));
  for (int din = 0; din < 3; din++)
    for (int cin = 0; cin < 3; cin++) {
      B2(ceed, b200_memset(unit, 0, usz));
      /* unit field (din, cin): Q-vector layout [elem][9][nq], component index din*3 + cin */
      B2(ceed, b200_fill_strided(unit + (size_t)(din * 3 + cin) * nq, 1.0, nq, (size_t)9 * nq, nelem));
      CeedChk(op_run_qfunction(op, nelem, nq, qin, qout));
      B2(ceed, b200_diag_accumulate(nelem, b->P, b->Q, b->d_interp1d, b->d_grad1d, din, cin, qout[oa], ediag));
    }
  double *l;
  CeedChk(vec_dev_rw(assembled, &l));
  CeedChk(rstr_apply_raw(r, 1, ediag, l));
  return 0;
}

/* Chunk tables for the host pipeline: elements in creation order, chunk boundaries on multiples of the
 * q-blocked group size; in_need = running max of the highest dof a chunk reads, out_final = lowest dof any
 * LATER chunk writes.  Any numbering gives correct tables; only (nearly) ordered ones let the stages overlap. */
static int rstr_pipe_setup(CeedElemRestriction r, int Q) {
  Ceed ceed = r->ceed;
  if (r->pipe_n != 0 && r->pipe_q == Q) return 0;
  r->pipe_q = Q;
  r->pipe_n = -1;
  const int EB = b200_elems_per_block(Q);
  int nch = r->nelem / B200_PIPE_MIN_ELEMS;
  /* measured on PCIe 5 x16, 2 x 407 MB: 1 chunk 15.9 ms, 4: 11.3, 8: 10.3, 16: 10.25, 32: 10.55 (duplex floor 8.9) */
  int maxch = B200_PIPE_CHUNKS;
  const char *env = getenv("CEED_B200_PIPE_CHUNKS"); /* tuning knob; 1 disables the pipeline */
  if (env && atoi(env) >= 1) maxch = atoi(env) < B200_PIPE_MAXC ? atoi(env) : B200_PIPE_MAXC;
  if (nch > maxch) nch = maxch;
  if (nch < 2) return 0;
  int per = (r->nelem + nch - 1) / nch;
  per = (per + EB - 1) / EB * EB;
  const size_t n = (size_t)r->nelem * r->elemsize;
  int *off = (int *)malloc(n * sizeof(int));
  if (!off) return CeedError(ceed, 3, "out of memory");
  B2(ceed, b200_memcpy_d2h(off, r->d_offsets, n * sizeof(int)));
  const long long span = (long long)(r->ncomp - 1) * r->compstride + 1;
  int c = 0;
  long long lo[B200_PIPE_MAXC], hi[B200_PIPE_MAXC];
  for (int e0 = 0; e0 < r->nelem; e0 += per, c++) {
    const int e1 = e0 + per < r->nelem ? e0 + per : r->nelem;
    long long l = r->lsize, h = 0;
    for (size_t i = (size_t)e0 * r->elemsize; i < (size_t)e1 * r->elemsize; i++) {
      if (off[i] < l) l = off[i];
      if (off[i] + span > h) h = off[i] + span;
    }
    lo[c] = l; hi[c] = h;
    r->pipe_end[c] = e1;
  }
  free(off);
  long long run = 0;
  for (int i = 0; i < c; i++) { if (hi[i] > run) run = hi[i]; r->pipe_in[i] = (size_t)run; }
  run = r->lsize;
  for (int i = c - 1; i >= 0; i--) { r->pipe_out[i] = (size_t)run; if (lo[i] < run) run = lo[i]; }
  r->pipe_n = c;
  return 0;
}

/* -memtype host fast path (matops.c:40-50 with host arrays): x current on the host only, y with a host array
 * attached, both page-locked, one fused operator -> pipelined copies and kernels.  Returns 1 in *done if taken. */
static int op_apply_hostpipe(CeedOperator op, CeedVector in, CeedVector out, int *done) {
  Ceed ceed = op->ceed;
  *done = 0;
  if (ceed->deterministic) return 0;  /* chunked launches scatter with atomics */
  if (op->kind != OP_FUSED_JACOBIAN && op->kind != OP_FUSED_RESIDUAL) return 0;
  if (!in || !out || in == out || !in->h_valid || in->d_valid || !in->h || !out->h) return 0;
  OpField *u = &op->in[op->ai];
  if (in->length != u->r->lsize || out->length != u->r->lsize) return 0;
  CeedChk(rstr_pipe_setup(u->r, u->b->Q));
  if (u->r->pipe_n < 2) return 0;
  if (!b200_host_is_pinned(in->h) || !b200_host_is_pinned(out->h)) return 0;
  b200_physics phys;
  CeedChk(qf_physics(op->qf, &phys));
  const int jac = op->kind == OP_FUSED_JACOBIAN;
  const double *qa;
  double *gu = NULL, *y;
  if (jac) CeedChk(jcache_get(op, &qa));
  else {
    CeedChk(vec_dev_read(op->in[1].v, &qa));
    if (op->problem != B200_PROB_LINELAS) CeedChk(vec_dev_write(op->out[1].v, &gu));
  }
  CeedChk(vec_alloc(in, CEED_MEM_DEVICE));
  CeedChk(vec_dev_write(out, &y));
  B2(ceed, b200_vec_set(y, 0.0, (size_t)out->length));
  B2(ceed, b200_apply_hostpipe(jac, op->problem, &phys, u->r->nelem, u->b->P, u->b->Q, u->b->interp1d, u->b->grad1d,
                               u->r->d_offsets, qa, gu, in->h, in->d, out->h, y, (size_t)out->length, u->r->pipe_n,
                               u->r->pipe_end, u->r->pipe_in, u->r->pipe_out));
  in->d_valid = 1;   /* whole of x was copied on the way */
  out->h_valid = 1;  /* whole of y is already in the caller's host array */
  *done = 1;
  return 0;
}

/* K12, K13, K14: the operator's program of the given kind, compiled with `compile` at its first use; *slot holds the
 * handle + 1 (0: not compiled yet).  K12 is compiled at the first apply (the point program of op_setup stays: it
 * reports source errors at set-up), K13 at the first CeedOperatorLinearAssemble, K14 at the first diagonal. */
typedef int (*jit_compile_fn)(const char *, const char *, const char *, int, const int *, int, const int *, int, int,
                              int, int, int *);
static int jit_op_handle(CeedOperator op, jit_compile_fn compile, int *slot, const char *what, int *h) {
  Ceed ceed = op->ceed;
  CeedQFunction qf = op->qf;
  if (!*slot) {
    int in_sizes[MAXF], out_sizes[MAXF], hh = -1;
    for (int i = 0; i < qf->nin; i++) in_sizes[i] = qf->in[i].size;
    for (int i = 0; i < qf->nout; i++) out_sizes[i] = qf->out[i].size;
    CeedBasis b = op->in[op->ai].b;
    if (compile(qf->jit_text, qf->jit_path, qf->name, qf->nin, in_sizes, qf->nout, out_sizes, op->ai, op->ao, b->P,
                b->Q, &hh))
      return CeedError(ceed, 1, "%s: %s of QFunction \"%s\" from %s: %s", CEED_B200_RESOURCE, what, qf->name,
                       qf->jit_path, b200_last_error());
    *slot = hh + 1;
  }
  *h = *slot - 1;
  return 0;
}

/* the device copies of a JIT operator's passive inputs (K12, K13, K14), from element e0 on; NULL at the active input */
static int jit_passive_inputs(CeedOperator op, int e0, const double **din) {
  CeedQFunction qf = op->qf;
  const int Q = op->in[op->ai].b->Q;
  for (int i = 0; i < qf->nin; i++) {
    din[i] = NULL;
    if (i == op->ai) continue;
    CeedChk(vec_dev_read(op->in[i].v, &din[i]));
    din[i] += (size_t)e0 * qf->in[i].size * Q * Q * Q;
  }
  return 0;
}

/* makes current what every element range of a fused apply reads, so that ranges can run on two streams at once: the
 * Jacobian cache of a built-in Jacobian (*jc); K12 of a JIT operator, compiled at its first apply (*h), with the device
 * copies of its passive vectors from element e0 on (din, dout).  A passive output the apply stores over all of its
 * entries (overwrite) is not copied in. */
static int op_fused_state(CeedOperator op, int e0, int overwrite, const double **jc, int *h, const double **din,
                          double **dout) {
  CeedQFunction qf = op->qf;
  if (op->kind == OP_FUSED_JACOBIAN) return jcache_get(op, jc);
  if (op->kind != OP_JIT_FUSED) return 0;
  const int Q = op->in[op->ai].b->Q;
  CeedChk(jit_op_handle(op, b200_jit_fused_compile, &op->jit_fused, "fused kernel", h));
  CeedChk(jit_passive_inputs(op, e0, din));
  for (int i = 0; i < qf->nout; i++) {
    dout[i] = NULL;
    if (i == op->ao) continue;
    if (overwrite) CeedChk(vec_dev_write(op->out[i].v, &dout[i]));
    else CeedChk(vec_dev_rw(op->out[i].v, &dout[i]));
    dout[i] += (size_t)e0 * qf->out[i].size * Q * Q * Q;
  }
  return 0;
}

/* the fused kernels on the element range [e0, e1), e0 a multiple of the q-blocked group size: the built-in residual or
 * Jacobian, or K12.  The active output is added to.  K12 stores its passive outputs (passive_add = 0, Apply) or adds to
 * them (ApplyAdd); the built-in residual always stores gradu. */
static int op_apply_range(CeedOperator op, CeedVector in, CeedVector out, int e0, int e1, int passive_add) {
  Ceed ceed = op->ceed;
  CeedQFunction qf = op->qf;
  OpField *u = &op->in[op->ai];
  const int P = u->b->P, Q = u->b->Q, P3 = P * P * P, Q3 = Q * Q * Q, nelem = u->r->nelem;
  const int whole = e0 == 0 && e1 == nelem;
  b200_physics phys;
  size_t bytes = 0;
  if (op->kind == OP_JIT_FUSED) CeedChk(jit_ctx_bytes(qf, &bytes));
  else CeedChk(qf_physics(qf, &phys));
  if (in->length < u->r->lsize || out->length < u->r->lsize)
    return CeedError(ceed, 1, "operator %s: active vectors shorter than the restriction's L-vector size %d", qf->name, u->r->lsize);
  if (ceed->deterministic && !whole)
    return CeedError(ceed, 1, "deterministic mode: element-range applies are not supported (the ordered sum runs over the whole restriction)");
  double *evec, *dout[MAXF], *y;
  const double *jc = NULL, *din[MAXF], *x;
  int h = -1;
  CeedChk(det_evec(ceed, u->r, &evec));
  CeedChk(op_fused_state(op, e0, !passive_add && whole, &jc, &h, din, dout));
  const double *qd = NULL;
  double *gu = NULL;
  if (op->kind == OP_FUSED_RESIDUAL) {
    CeedChk(vec_dev_read(op->in[1].v, &qd));
    qd += (size_t)e0 * 10 * Q3;
    if (op->problem != B200_PROB_LINELAS) {
      /* a partial range rewrites only its own slice of gradu: the rest must stay valid */
      if (whole) CeedChk(vec_dev_write(op->out[1].v, &gu));
      else CeedChk(vec_dev_rw(op->out[1].v, &gu));
      gu += (size_t)e0 * 9 * Q3;
    }
  }
  CeedChk(vec_dev_read(in, &x));
  CeedChk(vec_dev_rw(out, &y));
  const int *off = u->r->d_offsets + (size_t)e0 * P3;
  if (op->kind == OP_FUSED_RESIDUAL)
    B2(ceed, b200_apply_residual(op->problem, &phys, e1 - e0, P, Q, u->b->interp1d, u->b->grad1d, off, qd, gu, x, y,
                                 evec));
  else if (op->kind == OP_FUSED_JACOBIAN)
    B2(ceed, b200_apply_jacobian(op->problem, &phys, e1 - e0, P, Q, u->b->interp1d, u->b->grad1d, off,
                                 jc + (size_t)e0 * b200_jcache_ncomp(op->problem) * Q3, x, y, evec));
  else
    B2(ceed, b200_jit_fused_apply(h, qf->ctx, bytes, e1 - e0, u->b->interp1d, u->b->grad1d, off, x, y, evec, qf->nin,
                                  din, qf->nout, dout, passive_add));
  if (evec) CeedChk(rstr_ordered_add(u->r, 1, evec, y));
  return 0;
}

static int op_apply_add(CeedOperator op, CeedVector in, CeedVector out) {
  Ceed ceed = op->ceed;
  if (op->composite) {
    for (int i = 0; i < op->nsubs; i++) CeedChk(op_apply_add(op->subs[i], in, out));
    return 0;
  }
  if (op->kind == OP_UNSET) CeedChk(op_setup(op));
  if (op->kind == OP_GENERIC) return op_apply_generic(op, in, out);
  if (op->kind == OP_FUSED_TRANSFER) {
    const double *x;
    double *y;
    const int prolong = op->qf->in[0].emode == CEED_EVAL_INTERP;
    OpField *c = prolong ? &op->in[0] : &op->out[0], *f = prolong ? &op->out[0] : &op->in[0];
    CeedChk(vec_dev_read(in, &x));
    CeedChk(vec_dev_rw(out, &y));
    const double *mult = NULL;
    if (op->xfer_scale) {
      if (op->xfer_scale->length < f->r->lsize) return CeedError(ceed, 1, "transfer scaling vector shorter than the fine L-vector");
      CeedChk(vec_dev_read(op->xfer_scale, &mult));
    }
    const int inject = prolong && mult && op->xfer_inject;
    CeedElemRestriction ro = prolong ? f->r : c->r;
    double *evec = NULL;
    if (!inject) CeedChk(det_evec(ceed, ro, &evec));
    B2(ceed, b200_apply_transfer(!prolong, c->r->nelem, c->b->P, c->b->Q, c->b->interp1d, c->r->d_offsets, f->r->d_offsets,
                                 mult, inject, x, y, evec));
    if (evec) CeedChk(rstr_ordered_add(ro, 1, evec, y));
    return 0;
  }
  return op_apply_range(op, in, out, 0, op->in[op->ai].r->nelem, 1);
}

/* /gpu/b200 extension: ApplyAdd restricted to the elements [start, stop) of a fused residual / Jacobian operator
 * (creation order of the restriction).  Lets a partitioned caller run the elements that touch partition
 * interfaces first and overlap its halo exchange with the interior ones.  start must be a multiple of the
 * backend's element-group size (16 always is), and so must stop unless it is nelem: the kernels take the extent
 * of the range's last group from the range, while the q-blocked per-point vectors (qdata, Jacobian cache, gradu,
 * passive fields) lay out a group cut short by stop with the extent it has in the whole restriction. */
int CeedOperatorApplyAddRangeB200(CeedOperator op, CeedVector in, CeedVector out, CeedInt start, CeedInt stop) {
  Ceed ceed = op->ceed;
  if (op->composite) return CeedError(ceed, 1, "CeedOperatorApplyAddRangeB200: composite operators are not supported");
  if (op->kind == OP_UNSET) CeedChk(op_setup(op));
  if (!op_fused_apply(op))
    return CeedError(ceed, 1, "CeedOperatorApplyAddRangeB200: operator %s does not run on the fused kernels", op->qf->name);
  const int nelem = op->in[op->ai].r->nelem, EB = b200_elems_per_block(op->in[op->ai].b->Q);
  if (start < 0 || stop > nelem || start > stop || start % EB || (stop % EB && stop != nelem))
    return CeedError(ceed, 1, "CeedOperatorApplyAddRangeB200: bad element range [%d, %d) (nelem %d; start, and stop "
                     "unless it is nelem, must be multiples of %d)", start, stop, nelem, EB);
  if (start == stop) return 0;
  return op_apply_range(op, in, out, start, stop, 1);
}

/* /gpu/b200 extension for the p-multigrid transfer operators (Prolong_Ceed / Restrict_Ceed, matops.c:115-203): the
 * reference scales the fine vector by the inverse multiplicity in a separate VecPointwiseMult (:149 after the
 * prolongation, :176 before the restriction).  With a scaling vector set, the fused transfer kernel applies it on
 * the fly; inject != 0 additionally lets the prolongation STORE the interpolant at every fine node instead of
 * summing the element copies and dividing by their number (identical for a continuous coarse field).  Apply then
 * has overwrite semantics on the nodes it reaches.  scale == NULL restores the plain operator. */
int CeedOperatorSetTransferScalingB200(CeedOperator op, CeedVector scale, int inject) {
  Ceed ceed = op->ceed;
  if (op->composite) return CeedError(ceed, 1, "CeedOperatorSetTransferScalingB200: composite operator");
  if (op->kind == OP_UNSET) CeedChk(op_setup(op));
  if (op->kind != OP_FUSED_TRANSFER)
    return CeedError(ceed, 1, "CeedOperatorSetTransferScalingB200: operator %s is not a fused transfer operator", op->qf->name);
  if (scale) scale->refcount++;
  if (op->xfer_scale) CeedVectorDestroy(&op->xfer_scale);
  op->xfer_scale = scale;
  op->xfer_inject = scale ? inject : 0;
  return 0;
}

/* /gpu/b200 extension: the whole partitioned MatShell MatMult of ApplyLocalCeedOp (matops.c:26-60) in the masked
 * layout, issued from C in one call:
 *     out = 0;  out += A_loc in on the elements [0, n_interface) that touch a partition interface;
 *     halo exchange starts on its side stream (b200_halo_begin: interface partial sums are complete);
 *     out += A_loc in on the interior elements [n_interface, nelem)   -- overlaps the exchange;
 *     b200_halo_end: ordered sum of the holders' partial sums;  zero the Dirichlet rows d_mask[0..nmask).
 * halo may be NULL (single rank).  In deterministic mode (no element-range applies) the operator runs as a whole
 * and the exchange follows it. */
int CeedOperatorApplyPartitionedB200(CeedOperator op, CeedVector in, CeedVector out, CeedInt n_interface, void *halo,
                                     const CeedInt *d_mask, CeedInt nmask) {
  Ceed ceed = op->ceed;
  if (op->composite) return CeedError(ceed, 1, "CeedOperatorApplyPartitionedB200: composite operators are not supported");
  if (op->kind == OP_UNSET) CeedChk(op_setup(op));
  if (!op_fused_apply(op))
    return CeedError(ceed, 1, "CeedOperatorApplyPartitionedB200: operator %s does not run on the fused kernels", op->qf->name);
  const int nelem = op->in[op->ai].r->nelem, EB = b200_elems_per_block(op->in[op->ai].b->Q);
  if (n_interface < 0 || n_interface > nelem || (n_interface % EB && n_interface != nelem))
    return CeedError(ceed, 1, "CeedOperatorApplyPartitionedB200: n_interface %d must be a multiple of %d within [0, %d]", n_interface, EB, nelem);
  double *y;
  CeedChk(CeedVectorSetValue(out, 0.0));
  if (!halo || ceed->deterministic || n_interface == 0 || n_interface == nelem) {
    CeedChk(op_apply_range(op, in, out, 0, nelem, 0));
    CeedChk(vec_dev_rw(out, &y));
    if (halo) { B2(ceed, b200_halo_begin((b200_halo *)halo, y)); B2(ceed, b200_halo_end((b200_halo *)halo, y)); }
  } else {
    /* everything the two element ranges share is made current on the compute stream first (device copies of the
       vectors, the Jacobian cache, K12); then the interface elements + push run on the halo's high-priority side stream
       CONCURRENTLY with the interior elements on the compute stream (both only add into Y, on disjoint shared dofs) */
    const double *x, *jc, *din[MAXF];
    double *dout[MAXF];
    int h;
    CeedChk(vec_dev_read(in, &x));
    CeedChk(vec_dev_rw(out, &y));
    CeedChk(op_fused_state(op, 0, 0, &jc, &h, din, dout));
    void *side = NULL, *mainstream = b200_get_stream();
    B2(ceed, b200_halo_fork((b200_halo *)halo, &side));
    B2(ceed, b200_set_stream(side));
    int rc = op_apply_range(op, in, out, 0, n_interface, 0);
    b200_set_stream(mainstream);
    if (rc) return rc;
    B2(ceed, b200_halo_begin_forked((b200_halo *)halo, y));
    CeedChk(op_apply_range(op, in, out, n_interface, nelem, 0));
    B2(ceed, b200_halo_end((b200_halo *)halo, y));
  }
  if (nmask > 0) B2(ceed, b200_mask_zero(y, d_mask, (size_t)nmask));
  return 0;
}

/* libCEED interface semantics: zero every output (active and passive), then ApplyAdd */
int CeedOperatorApplyAdd(CeedOperator op, CeedVector in, CeedVector out, CeedRequest *request) {
  (void)request;
  CeedChk(op_apply_add(op, in, out));
  return vec_write_through(out);
}
static int op_apply(CeedOperator op, CeedVector in, CeedVector out) {
  if (op->composite) {
    if (out && out != CEED_VECTOR_NONE) CeedChk(CeedVectorSetValue(out, 0.0));
    for (int i = 0; i < op->nsubs; i++) CeedChk(op_apply_add(op->subs[i], in, out));
    return 0;
  }
  if (op->kind == OP_UNSET) CeedChk(op_setup(op));
  {
    int done = 0;
    CeedChk(op_apply_hostpipe(op, in, out, &done));
    if (done) return 0;
  }
  for (int i = 0; i < op->qf->nout; i++) {
    CeedVector v = op->out[i].v == CEED_VECTOR_ACTIVE ? out : op->out[i].v;
    if (!v || v == CEED_VECTOR_NONE) continue;
    /* the fused residual kernel overwrites every entry of its passive output (gradu) itself */
    if (op->kind == OP_FUSED_RESIDUAL && i == 1) continue;
    if (op->kind == OP_JIT_FUSED && i != op->ao) continue;  /* K12 stores them (passive_add = 0 below) */
    CeedChk(CeedVectorSetValue(v, 0.0));
  }
  if (op_fused_apply(op)) return op_apply_range(op, in, out, 0, op->in[op->ai].r->nelem, 0);
  return op_apply_add(op, in, out);
}
int CeedOperatorApply(CeedOperator op, CeedVector in, CeedVector out, CeedRequest *request) {
  (void)request;
  CeedChk(op_apply(op, in, out));
  return vec_write_through(out);
}

/* the diagonal of a fused Jacobian, added to `assembled`: K3 from the built-in Jacobian cache, or K14 around the user
 * function (compiled at the operator's first diagonal; linear in its active input, as every Jacobian QFunction is),
 * which reads the passive inputs where K12 reads them and never writes the passive outputs.  Both add at the
 * restriction's offsets, so the vector must hold its whole L-vector. */
static int op_diagonal_fused(CeedOperator op, CeedVector assembled) {
  Ceed ceed = op->ceed;
  CeedQFunction qf = op->qf;
  OpField *u = &op->in[op->ai];
  if (assembled->length < u->r->lsize)
    return CeedError(ceed, 1, "CeedOperatorLinearAssembleDiagonal: operator %s: vector shorter than the restriction's "
                              "L-vector size %d", qf->name, u->r->lsize);
  b200_physics phys;
  const double *jc, *din[MAXF];
  size_t bytes;
  int h;
  if (op->kind == OP_JIT_FUSED) {
    CeedChk(jit_op_handle(op, b200_jit_diag_compile, &op->jit_diag, "diagonal kernel", &h));
    CeedChk(jit_ctx_bytes(qf, &bytes));
    CeedChk(jit_passive_inputs(op, 0, din));
  } else {
    CeedChk(qf_physics(qf, &phys));
    CeedChk(jcache_get(op, &jc));
  }
  double *d, *evec;
  CeedChk(vec_dev_rw(assembled, &d));
  CeedChk(det_evec(ceed, u->r, &evec));
  if (op->kind == OP_JIT_FUSED)
    B2(ceed, b200_jit_diag_apply(h, qf->ctx, bytes, u->r->nelem, u->b->interp1d, u->b->grad1d, u->r->d_offsets, qf->nin,
                                 din, d, evec));
  else
    B2(ceed, b200_apply_diagonal(op->problem, &phys, u->r->nelem, u->b->P, u->b->Q, u->b->interp1d, u->b->grad1d,
                                 u->r->d_offsets, jc, d, evec));
  if (evec) CeedChk(rstr_ordered_add(u->r, 1, evec, d));
  return 0;
}

int CeedOperatorLinearAssembleAddDiagonal(CeedOperator op, CeedVector assembled, CeedRequest *request) {
  (void)request;
  if (op->composite) {
    for (int i = 0; i < op->nsubs; i++) CeedChk(CeedOperatorLinearAssembleAddDiagonal(op->subs[i], assembled, request));
    return 0;
  }
  if (op->kind == OP_UNSET) CeedChk(op_setup(op));
  if (!op_fused_jacobian(op)) return op_diagonal_generic(op, assembled);
  return op_diagonal_fused(op, assembled);
}
int CeedOperatorLinearAssembleDiagonal(CeedOperator op, CeedVector assembled, CeedRequest *request) {
  CeedChk(CeedVectorSetValue(assembled, 0.0));
  return CeedOperatorLinearAssembleAddDiagonal(op, assembled, request);
}

/* COO assembly: entry (e, col, row) of element e sits at (e*24 + col)*24 + row, element dof = node*3 + comp.
 * Built-in fused Jacobians: K8 from the Jacobian cache.  JIT operators on K12 (OP_JIT_FUSED): K13 around the user
 * function, which must be linear in its active input (every Jacobian QFunction is). */
static int op_assemblable(CeedOperator op) {
  Ceed ceed = op->ceed;
  if (op->composite) return CeedError(ceed, 1, "CeedOperatorLinearAssemble: composite operators are not supported by /gpu/b200");
  if (op->kind == OP_UNSET) CeedChk(op_setup(op));
  if (op->kind == OP_GENERIC && op->qf->jit_handle >= 0) {
    CeedBasis b = NULL;
    for (int i = 0; i < op->qf->nin && !b; i++)
      if (op->in[i].v == CEED_VECTOR_ACTIVE && op->in[i].b != CEED_BASIS_COLLOCATED) b = op->in[i].b;
    return CeedError(ceed, 1, "CeedOperatorLinearAssemble: JIT QFunction %s runs on the generic path: its fields are "
                              "not of the fused shape or its basis (P, Q) = (%d, %d) has no fused kernel, and /gpu/b200 "
                              "assembles only operators of the fused kernels; there is no CPU fallback",
                     op->qf->name, b ? b->P : 0, b ? b->Q : 0);
  }
  CeedBasis b = op->in[op->ai].b;
  if (!op_fused_jacobian(op) || b->P != 2)
    return CeedError(ceed, 1, "CeedOperatorLinearAssemble: /gpu/b200 assembles fused Jacobian operators on a trilinear "
                              "(P = 2) level only (operator %s, P = %d); there is no CPU fallback",
                     op->qf->name, b ? b->P : 0);
  return 0;
}

int CeedOperatorLinearAssembleSymbolic(CeedOperator op, CeedInt *num_entries, CeedInt **rows, CeedInt **cols) {
  Ceed ceed = op->ceed;
  CeedChk(op_assemblable(op));
  CeedElemRestriction r = op->in[op->ai].r;
  const size_t nelem = (size_t)r->nelem, ne = nelem * 576;
  if (ne > 2147483647u) return CeedError(ceed, 1, "CeedOperatorLinearAssembleSymbolic: %zu entries overflow CeedInt", ne);
  int *off = (int *)malloc(sizeof(int) * (nelem * 8 + 1));
  *rows = (CeedInt *)malloc(sizeof(CeedInt) * (ne + 1));
  *cols = (CeedInt *)malloc(sizeof(CeedInt) * (ne + 1));
  if (!off || !*rows || !*cols) { free(off); free(*rows); free(*cols); return CeedError(ceed, 3, "out of memory"); }
  if (nelem) B2(ceed, b200_memcpy_d2h(off, r->d_offsets, sizeof(int) * nelem * 8));
  for (size_t e = 0; e < nelem; e++)
    for (int c = 0; c < 24; c++)
      for (int w = 0; w < 24; w++) {
        (*rows)[(e * 24 + c) * 24 + w] = off[e * 8 + w / 3] + (w % 3) * r->compstride;
        (*cols)[(e * 24 + c) * 24 + w] = off[e * 8 + c / 3] + (c % 3) * r->compstride;
      }
  free(off);
  *num_entries = (CeedInt)ne;
  return 0;
}

/* K13: compile the assembly program at the first CeedOperatorLinearAssemble, then assemble; the operator's vectors
 * are only read (passive outputs are never written) */
static int op_assemble_jit(CeedOperator op, double *v) {
  Ceed ceed = op->ceed;
  CeedQFunction qf = op->qf;
  OpField *u = &op->in[op->ai];
  int h;
  size_t bytes;
  CeedChk(jit_op_handle(op, b200_jit_assemble_compile, &op->jit_assemble, "assembly kernel", &h));
  CeedChk(jit_ctx_bytes(qf, &bytes));
  const double *din[MAXF];
  CeedChk(jit_passive_inputs(op, 0, din));
  B2(ceed, b200_jit_assemble_apply(h, qf->ctx, bytes, u->r->nelem, u->b->interp1d, u->b->grad1d,
                                   qf->nin, din, v));
  return 0;
}

int CeedOperatorLinearAssemble(CeedOperator op, CeedVector values) {
  Ceed ceed = op->ceed;
  CeedChk(op_assemblable(op));
  OpField *u = &op->in[op->ai];
  if ((size_t)values->length < (size_t)u->r->nelem * 576)
    return CeedError(ceed, 1, "CeedOperatorLinearAssemble: values vector holds %d entries, %zu needed", values->length,
                     (size_t)u->r->nelem * 576);
  double *v;
  if (op->kind == OP_JIT_FUSED) {
    CeedChk(vec_dev_write(values, &v));
    return op_assemble_jit(op, v);
  }
  b200_physics phys;
  CeedChk(qf_physics(op->qf, &phys));
  const double *jc;
  CeedChk(jcache_get(op, &jc));
  CeedChk(vec_dev_write(values, &v));
  B2(ceed, b200_assemble_p1(op->problem, &phys, u->r->nelem, u->b->Q, u->b->interp1d, u->b->grad1d, jc, v));
  return 0;
}

int CeedOperatorDestroy(CeedOperator *op) {
  if (!op || !*op) return 0;
  CeedOperator o = *op;
  *op = NULL;
  if (--o->refcount > 0) return 0;
  if (o->composite) {
    for (int i = 0; i < o->nsubs; i++) CeedOperatorDestroy(&o->subs[i]);
  } else {
    for (int i = 0; i < 2 * MAXF; i++) {
      OpField *f = i < MAXF ? &o->in[i] : &o->out[i - MAXF];
      if (f->set) {
        CeedElemRestriction r = f->r; CeedBasis b = f->b; CeedVector v = f->v;
        if (r && r != CEED_ELEMRESTRICTION_NONE) CeedElemRestrictionDestroy(&r);
        if (b && b != CEED_BASIS_COLLOCATED) CeedBasisDestroy(&b);
        if (v && v != CEED_VECTOR_ACTIVE && v != CEED_VECTOR_NONE) CeedVectorDestroy(&v);
      }
      b200_free(o->ebuf[i]);
      b200_free(o->qbuf[i]);
    }
    CeedQFunctionDestroy(&o->qf);
    if (o->xfer_scale) CeedVectorDestroy(&o->xfer_scale);
  }
  Ceed c = o->ceed;
  free(o);
  return CeedDestroy(&c);
}
