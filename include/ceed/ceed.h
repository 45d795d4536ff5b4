/* ceed.h -- the libCEED user API subset that the reference mini-app calls, served by the
 * B200-native backend resource "/gpu/b200" (libceed_b200.so).
 *
 * The reference (ArashMehraban/CeedPetscSolid) links against upstream libCEED, which is NOT
 * vendored in it.  This header reproduces exactly the API surface its sources use
 * (SURVEY.md Appendix A; call-site citations below are /root/reference paths), with
 * upstream's names, argument meaning and enum values, so that src/setuplibceed.c,
 * src/matops.c, src/misc.c and elasticity.c compile against it unchanged.  When a real
 * libCEED is present the same backend registers into it instead (INTEGRATION.md).
 *
 * All functions return int (0 = success).  The reference never checks those codes
 * (e.g. src/matops.c:40-50), so errors go through the Ceed's error handler; the default
 * handler prints and aborts like upstream's.
 */
#ifndef CEED_B200_CEED_H
#define CEED_B200_CEED_H

#include <stdarg.h>
#include <stddef.h>
#include <stdint.h>
#include <stdio.h>

#ifdef __cplusplus
#define CEED_EXTERN extern "C"
#else
#define CEED_EXTERN extern
#endif

typedef int32_t CeedInt;
typedef double CeedScalar;

typedef struct Ceed_private *Ceed;
typedef struct CeedRequest_private *CeedRequest;
typedef struct CeedVector_private *CeedVector;
typedef struct CeedElemRestriction_private *CeedElemRestriction;
typedef struct CeedBasis_private *CeedBasis;
typedef struct CeedQFunction_private *CeedQFunction;
typedef struct CeedOperator_private *CeedOperator;

typedef enum { CEED_MEM_HOST = 0, CEED_MEM_DEVICE = 1 } CeedMemType;
typedef enum { CEED_COPY_VALUES = 0, CEED_USE_POINTER = 1, CEED_OWN_POINTER = 2 } CeedCopyMode;
typedef enum { CEED_NORM_1 = 0, CEED_NORM_2 = 1, CEED_NORM_MAX = 2 } CeedNormType;
typedef enum { CEED_NOTRANSPOSE = 0, CEED_TRANSPOSE = 1 } CeedTransposeMode;
typedef enum {
  CEED_EVAL_NONE = 0,
  CEED_EVAL_INTERP = 1,
  CEED_EVAL_GRAD = 2,
  CEED_EVAL_DIV = 4,
  CEED_EVAL_CURL = 8,
  CEED_EVAL_WEIGHT = 16
} CeedEvalMode;
typedef enum { CEED_GAUSS = 0, CEED_GAUSS_LOBATTO = 1 } CeedQuadMode;

CEED_EXTERN const char *const CeedMemTypes[];   /* printed at elasticity.c:316-318 */
CEED_EXTERN const char *const CeedEvalModes[];

/* sentinels (setuplibceed.c:304-318,378-386,529-539) */
CEED_EXTERN const CeedInt CEED_STRIDES_BACKEND[3];
CEED_EXTERN const CeedBasis CEED_BASIS_COLLOCATED;
CEED_EXTERN const CeedVector CEED_VECTOR_ACTIVE;
CEED_EXTERN const CeedVector CEED_VECTOR_NONE;
CEED_EXTERN const CeedElemRestriction CEED_ELEMRESTRICTION_NONE;
CEED_EXTERN const CeedQFunction CEED_QFUNCTION_NONE;
CEED_EXTERN CeedRequest *const CEED_REQUEST_IMMEDIATE;
CEED_EXTERN CeedRequest *const CEED_REQUEST_ORDERED;

/* ---- QFunction source macros (the reference's qfunctions headers) ------------------------------------ */
#ifndef CEED_QFUNCTION
#define CEED_QFUNCTION(name)                            \
  static const char name##_loc[] = __FILE__ ":" #name;  \
  static int name
#endif
#ifndef CEED_Q_VLA
#define CEED_Q_VLA Q
#endif
#ifndef CeedPragmaSIMD
#if defined(_OPENMP)
#define CeedPragmaSIMD _Pragma("omp simd")
#else
#define CeedPragmaSIMD
#endif
#endif

typedef int (*CeedQFunctionUser)(void *ctx, const CeedInt Q, const CeedScalar *const *in, CeedScalar *const *out);

/* ---- Ceed (elasticity.c:110-116,308,897) ------------------------------------------ */
CEED_EXTERN int CeedInit(const char *resource, Ceed *ceed);
CEED_EXTERN int CeedDestroy(Ceed *ceed);
CEED_EXTERN int CeedGetResource(Ceed ceed, const char **resource);
CEED_EXTERN int CeedGetPreferredMemType(Ceed ceed, CeedMemType *type);
CEED_EXTERN int CeedIsDeterministic(Ceed ceed, int *isDeterministic);

/* error handling: upstream's CeedError / handlers */
typedef int (*CeedErrorHandler)(Ceed, const char *file, int line, const char *func, int ecode,
                                const char *format, va_list *args);
CEED_EXTERN int CeedErrorAbort(Ceed, const char *, int, const char *, int, const char *, va_list *);
CEED_EXTERN int CeedErrorReturn(Ceed, const char *, int, const char *, int, const char *, va_list *);
CEED_EXTERN int CeedErrorStore(Ceed, const char *, int, const char *, int, const char *, va_list *);
CEED_EXTERN int CeedSetErrorHandler(Ceed ceed, CeedErrorHandler handler);
CEED_EXTERN int CeedGetErrorMessage(Ceed ceed, const char **errmsg);
CEED_EXTERN int CeedResetErrorMessage(Ceed ceed, const char **errmsg);

/* ---- CeedVector (matops.c:40-50; setuplibceed.c:327-329,355-361,627-636) ----------- */
CEED_EXTERN int CeedVectorCreate(Ceed ceed, CeedInt len, CeedVector *vec);
CEED_EXTERN int CeedVectorSetArray(CeedVector vec, CeedMemType mtype, CeedCopyMode cmode, CeedScalar *array);
CEED_EXTERN int CeedVectorTakeArray(CeedVector vec, CeedMemType mtype, CeedScalar **array);
CEED_EXTERN int CeedVectorSetValue(CeedVector vec, CeedScalar value);
CEED_EXTERN int CeedVectorSyncArray(CeedVector vec, CeedMemType mtype);
CEED_EXTERN int CeedVectorGetArray(CeedVector vec, CeedMemType mtype, CeedScalar **array);
CEED_EXTERN int CeedVectorGetArrayRead(CeedVector vec, CeedMemType mtype, const CeedScalar **array);
CEED_EXTERN int CeedVectorRestoreArray(CeedVector vec, CeedScalar **array);
CEED_EXTERN int CeedVectorRestoreArrayRead(CeedVector vec, const CeedScalar **array);
CEED_EXTERN int CeedVectorNorm(CeedVector vec, CeedNormType type, CeedScalar *norm);
CEED_EXTERN int CeedVectorReciprocal(CeedVector vec);
CEED_EXTERN int CeedVectorGetLength(CeedVector vec, CeedInt *length);
CEED_EXTERN int CeedVectorDestroy(CeedVector *vec);

/* ---- CeedElemRestriction (setuplibceed.c:235,304-318,326,626; misc.c:123) ---------- */
CEED_EXTERN int CeedElemRestrictionCreate(Ceed ceed, CeedInt nelem, CeedInt elemsize, CeedInt ncomp,
                                          CeedInt compstride, CeedInt lsize, CeedMemType mtype,
                                          CeedCopyMode cmode, const CeedInt *offsets, CeedElemRestriction *rstr);
CEED_EXTERN int CeedElemRestrictionCreateStrided(Ceed ceed, CeedInt nelem, CeedInt elemsize, CeedInt ncomp,
                                                 CeedInt lsize, const CeedInt strides[3], CeedElemRestriction *rstr);
CEED_EXTERN int CeedElemRestrictionCreateVector(CeedElemRestriction rstr, CeedVector *lvec, CeedVector *evec);
CEED_EXTERN int CeedElemRestrictionApply(CeedElemRestriction rstr, CeedTransposeMode tmode, CeedVector u,
                                         CeedVector ru, CeedRequest *request);
CEED_EXTERN int CeedElemRestrictionGetMultiplicity(CeedElemRestriction rstr, CeedVector mult);
CEED_EXTERN int CeedElemRestrictionGetNumElements(CeedElemRestriction rstr, CeedInt *numelem);
CEED_EXTERN int CeedElemRestrictionGetElementSize(CeedElemRestriction rstr, CeedInt *elemsize);
CEED_EXTERN int CeedElemRestrictionGetLVectorSize(CeedElemRestriction rstr, CeedInt *lsize);
CEED_EXTERN int CeedElemRestrictionGetNumComponents(CeedElemRestriction rstr, CeedInt *ncomp);
CEED_EXTERN int CeedElemRestrictionDestroy(CeedElemRestriction *rstr);

/* ---- CeedBasis (setuplibceed.c:335-353,782-803) ------------------------------------ */
CEED_EXTERN int CeedBasisCreateTensorH1Lagrange(Ceed ceed, CeedInt dim, CeedInt ncomp, CeedInt P, CeedInt Q,
                                                CeedQuadMode qmode, CeedBasis *basis);
CEED_EXTERN int CeedBasisCreateTensorH1(Ceed ceed, CeedInt dim, CeedInt ncomp, CeedInt P1d, CeedInt Q1d,
                                        const CeedScalar *interp1d, const CeedScalar *grad1d,
                                        const CeedScalar *qref1d, const CeedScalar *qweight1d, CeedBasis *basis);
CEED_EXTERN int CeedBasisApply(CeedBasis basis, CeedInt nelem, CeedTransposeMode tmode, CeedEvalMode emode,
                               CeedVector u, CeedVector v);
CEED_EXTERN int CeedBasisGetNumNodes(CeedBasis basis, CeedInt *P);
CEED_EXTERN int CeedBasisGetNumQuadraturePoints(CeedBasis basis, CeedInt *Q);
CEED_EXTERN int CeedBasisGetInterp1D(CeedBasis basis, const CeedScalar **interp1d);
CEED_EXTERN int CeedBasisGetGrad1D(CeedBasis basis, const CeedScalar **grad1d);
CEED_EXTERN int CeedBasisGetQRef(CeedBasis basis, const CeedScalar **qref);
CEED_EXTERN int CeedBasisGetQWeights(CeedBasis basis, const CeedScalar **qweight);
CEED_EXTERN int CeedBasisDestroy(CeedBasis *basis);
CEED_EXTERN int CeedGaussQuadrature(CeedInt Q, CeedScalar *qref1d, CeedScalar *qweight1d);
CEED_EXTERN int CeedLobattoQuadrature(CeedInt Q, CeedScalar *qref1d, CeedScalar *qweight1d);

/* ---- CeedQFunction (setuplibceed.c:370-377,518-526,818-826; elasticity.c:249-252) --- */
CEED_EXTERN int CeedQFunctionCreateInterior(Ceed ceed, CeedInt vlength, CeedQFunctionUser f, const char *source,
                                            CeedQFunction *qf);
CEED_EXTERN int CeedQFunctionCreateIdentity(Ceed ceed, CeedInt size, CeedEvalMode inmode, CeedEvalMode outmode,
                                            CeedQFunction *qf);
CEED_EXTERN int CeedQFunctionAddInput(CeedQFunction qf, const char *fieldname, CeedInt size, CeedEvalMode emode);
CEED_EXTERN int CeedQFunctionAddOutput(CeedQFunction qf, const char *fieldname, CeedInt size, CeedEvalMode emode);
CEED_EXTERN int CeedQFunctionSetContext(CeedQFunction qf, void *ctx, size_t ctxsize);
CEED_EXTERN int CeedQFunctionDestroy(CeedQFunction *qf);

/* ---- CeedOperator (matops.c:46,138,187,227; setuplibceed.c:378-393,529-542,829-863) - */
CEED_EXTERN int CeedOperatorCreate(Ceed ceed, CeedQFunction qf, CeedQFunction dqf, CeedQFunction dqfT,
                                   CeedOperator *op);
CEED_EXTERN int CeedCompositeOperatorCreate(Ceed ceed, CeedOperator *op);
CEED_EXTERN int CeedCompositeOperatorAddSub(CeedOperator compositeop, CeedOperator subop);
CEED_EXTERN int CeedOperatorSetField(CeedOperator op, const char *fieldname, CeedElemRestriction r, CeedBasis b,
                                     CeedVector v);
CEED_EXTERN int CeedOperatorApply(CeedOperator op, CeedVector in, CeedVector out, CeedRequest *request);
CEED_EXTERN int CeedOperatorApplyAdd(CeedOperator op, CeedVector in, CeedVector out, CeedRequest *request);
CEED_EXTERN int CeedOperatorLinearAssembleDiagonal(CeedOperator op, CeedVector assembled, CeedRequest *request);
CEED_EXTERN int CeedOperatorLinearAssembleAddDiagonal(CeedOperator op, CeedVector assembled, CeedRequest *request);
/* full assembly in COO form (upstream libCEED >= 0.8; what PETSc's MatSetPreallocationCOO/MatSetValuesCOO consume):
 * Symbolic returns malloc'ed host arrays the caller frees; values is a CeedVector of num_entries doubles.
 * /gpu/b200 implements both for fused Jacobian operators on a trilinear (P = 2) level -- the coarse level of the
 * reference's p-multigrid -- and raises an error otherwise. */
CEED_EXTERN int CeedOperatorLinearAssembleSymbolic(CeedOperator op, CeedInt *num_entries, CeedInt **rows, CeedInt **cols);
CEED_EXTERN int CeedOperatorLinearAssemble(CeedOperator op, CeedVector values);
CEED_EXTERN int CeedOperatorDestroy(CeedOperator *op);

/* ---- /gpu/b200 extensions (not part of upstream; used by the harness and the tests) -- */
/* 1 if the operator's Apply runs as ONE fused kernel (gather..scatter), 0 if generic */
/* ApplyAdd on the element range [start, stop) of a fused operator (halo-exchange overlap in partitioned runs); start,
 * and stop unless it is the element count, must be multiples of the backend's element-group size (16 always is) */
CEED_EXTERN int CeedOperatorApplyAddRangeB200(CeedOperator op, CeedVector in, CeedVector out, CeedInt start, CeedInt stop);
/* the partitioned MatMult of ApplyLocalCeedOp (matops.c:26-60) in one call: interface elements, halo exchange
 * (b200_halo handle, include/b200_kernels.h; NULL = none) overlapped with the interior elements, Dirichlet rows zeroed */
CEED_EXTERN int CeedOperatorApplyPartitionedB200(CeedOperator op, CeedVector in, CeedVector out, CeedInt n_interface,
                                                 void *halo, const CeedInt *d_mask, CeedInt nmask);
/* fused p-multigrid transfer operators: apply the fine-side inverse-multiplicity scaling of Prolong_Ceed /
 * Restrict_Ceed (matops.c:149,176) inside the kernel; inject != 0: the prolongation stores the interpolant */
CEED_EXTERN int CeedOperatorSetTransferScalingB200(CeedOperator op, CeedVector scale, int inject);
CEED_EXTERN int CeedOperatorIsFusedB200(CeedOperator op, int *isFused);
/* 1 if the operator's Apply runs as ONE kernel generated around its JIT-compiled user QFunction ("/gpu/b200:jit", K12);
 * such operators report 0 from CeedOperatorIsFusedB200, which means "runs on a built-in fused kernel" */
CEED_EXTERN int CeedOperatorIsJitFusedB200(CeedOperator op, int *isJitFused);
/* kernels launched by this library since the last reset (bench.py "gpu_launches") */
CEED_EXTERN unsigned long long CeedB200LaunchCount(void);
CEED_EXTERN void CeedB200LaunchCountReset(void);
/* run the backend on a caller-owned cudaStream_t instead of the legacy default stream */
CEED_EXTERN int CeedB200SetStream(Ceed ceed, void *cuda_stream);
CEED_EXTERN int CeedB200Synchronize(Ceed ceed);

#endif /* CEED_B200_CEED_H */
