/* b200_kernels.h -- thin C-ABI over the hand-written sm_100a CUDA kernels of the
 * `/gpu/b200` libCEED backend.  Plain pointers and sizes only (no CUDA, torch or C++
 * types), so the backend proper (csrc/ceed_b200.c) is C99 and any host language can
 * bind these entry points directly.
 *
 * Every function returns 0 on success or a CUDA error code (!= 0); b200_last_error()
 * gives the message.  All device work is issued on the stream set with
 * b200_set_stream() (default: the legacy default stream 0, which orders against PETSc
 * VecCUDA kernels as SURVEY.md 8(b) "Threading / streams" requires).
 *
 * Each group cites the reference interface it replaces; libCEED itself is not vendored
 * in the reference, its call sites are.
 */
#ifndef B200_KERNELS_H
#define B200_KERNELS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- problem / QFunction identifiers --------------------------------------------- */
/* problemOptions[] /root/reference/src/setuplibceed.c:41-107 */
enum { B200_PROB_LINELAS = 0, B200_PROB_HYPERSS = 1, B200_PROB_HYPERFS = 2 };

/* user QFunctions recognised by name (the "<file>:<Name>" locator given to
 * CeedQFunctionCreateInterior, setuplibceed.c:370,518,818) + the gallery Identity
 * (elasticity.c:249-252) */
enum {
  B200_QF_NONE = 0,
  B200_QF_SETUPGEO,    /* qfunctions/common.h:47  */
  B200_QF_LINELAS_F,   /* qfunctions/linElas.h:39 */
  B200_QF_LINELAS_DF,  /* qfunctions/linElas.h:163 */
  B200_QF_HYPERSS_F,   /* qfunctions/hyperSS.h:60 */
  B200_QF_HYPERSS_DF,  /* qfunctions/hyperSS.h:187 */
  B200_QF_HYPERFS_F,   /* qfunctions/hyperFS.h:147 */
  B200_QF_HYPERFS_DF,  /* qfunctions/hyperFS.h:286 */
  B200_QF_IDENTITY,    /* libCEED gallery "Identity" */
  B200_QF_CONST_FORCE, /* qfunctions/constantForce.h:39   SetupConstantForce */
  B200_QF_MMS_FORCE,   /* qfunctions/manufacturedForce.h:39 SetupMMSForce    */
  B200_QF_MMS_TRUE,    /* qfunctions/manufacturedTrue.h:30  MMSTrueSoln      */
  /* one-shot post-processing (setuplibceed.c:650-737): in = (du GRAD, qdata) -> energy (1);
   * in = (u INTERP, du GRAD, qdata) -> diagnostic (8) = u, pressure, 2 invariants, volume ratio, energy density */
  B200_QF_LINELAS_ENERGY,  /* qfunctions/linElas.h:285 */
  B200_QF_HYPERSS_ENERGY,  /* qfunctions/hyperSS.h:326 */
  B200_QF_HYPERFS_ENERGY,  /* qfunctions/hyperFS.h:469 */
  B200_QF_LINELAS_DIAG,    /* qfunctions/linElas.h:376 */
  B200_QF_HYPERSS_DIAG,    /* qfunctions/hyperSS.h:418 */
  B200_QF_HYPERFS_DIAG,    /* qfunctions/hyperFS.h:559 */
  B200_QF_LAST = B200_QF_HYPERFS_DIAG
};

/* Physics_private {nu, E}  /root/reference/elasticity.h:30-37 */
typedef struct { double nu, E; } b200_physics;

/* ---- device / memory -------------------------------------------------------------- */
int b200_device_count(int *count);
int b200_set_device(int dev);
int b200_get_device(int *dev);
int b200_set_stream(void *cuda_stream);          /* cudaStream_t, NULL = legacy default */
void *b200_get_stream(void);
int b200_sync(void);                             /* synchronise the backend stream */
const char *b200_last_error(void);
int b200_device_name(char *buf, int len);
int b200_sm_count(int *count);

int b200_malloc(void **dptr, size_t bytes);
int b200_free(void *dptr);
int b200_malloc_host(void **hptr, size_t bytes); /* pinned */
int b200_free_host(void *hptr);
int b200_memset(void *dptr, int value, size_t bytes);
int b200_memcpy_h2d(void *d, const void *h, size_t bytes);
int b200_memcpy_d2h(void *h, const void *d, size_t bytes);   /* synchronises */
int b200_memcpy_d2d(void *d, const void *s, size_t bytes);
int b200_pointer_is_device(const void *p, int *is_device);

/* launch counter: number of kernels of THIS library launched since the last reset */
unsigned long long b200_launch_count(void);
void b200_launch_count_reset(void);

/* ---- CeedVector kernels (matops.c:34,56,149,176; misc.c:119-143) ------------------- */
int b200_vec_set(double *d, double value, size_t n);
int b200_vec_reciprocal(double *d, size_t n);
int b200_vec_scale(double *d, double alpha, size_t n);
int b200_vec_axpy(double *y, double alpha, const double *x, size_t n);            /* y += a x   */
int b200_vec_aypx(double *y, double alpha, const double *x, size_t n);            /* y = x + a y */
int b200_vec_axpby(double *z, double a, const double *x, double b, const double *y, size_t n);
int b200_vec_pointwise_mult(double *w, const double *x, const double *y, size_t n);
int b200_vec_dot(const double *x, const double *y, size_t n, double *dresult);    /* device scalar */
int b200_vec_dot_weighted(const double *w, const double *x, const double *y, size_t n, double *dresult); /* sum (w x) y */
int b200_vec_dot_host(const double *x, const double *y, size_t n, double *hresult);
int b200_vec_norm_host(const double *x, size_t n, int norm_type, double *hresult); /* 0=1,1=2,2=max */
/* index gather / scatter used by the halo exchange and the global<->local maps
 * (DMGlobalToLocal / DMLocalToGlobal, matops.c:33,57) */
int b200_gather(double *dst, const double *src, const int *idx, size_t n);        /* dst[i]=src[idx[i]] */
int b200_scatter_set(double *dst, const int *idx, const double *src, size_t n);   /* dst[idx[i]]=src[i] */
int b200_scatter_add(double *dst, const int *idx, const double *src, size_t n);   /* dst[idx[i]]+=src[i] */
int b200_mask_zero(double *d, const int *idx, size_t n);                          /* d[idx[i]] = 0 */
/* VecZeroEntries(Xloc) + DMGlobalToLocal(INSERT) in one pass (matops.c:106,33):
 * dst[i] = idx[i] >= 0 ? src[idx[i]] : 0  (idx = local dof -> global dof, -1 for ghost / Dirichlet dofs) */
int b200_gather_or_zero(double *dst, const double *src, const int *idx, size_t n);
/* dst[i] = src[idx[i]] where idx[i] >= 0, dst[i] untouched elsewhere (masked layouts: free dofs only) */
int b200_copy_where(double *dst, const double *src, const int *idx, size_t n);
/* BLAS-1 with DEVICE scalars (alpha = sign * num[0] / den[0]) and a fused CG update
 *   x += alpha p,  r -= alpha Ap,  z = dinv .* r   (alpha = rz[0] / pAp[0])
 * so that a Krylov loop (the coarse-level solve) runs without a host synchronisation per dot product */
int b200_vec_axpy_dev(double *y, const double *x, size_t n, const double *num, const double *den, double sign);
int b200_vec_aypx_dev(double *y, const double *x, size_t n, const double *num, const double *den);
int b200_pcg_update(double *x, double *r, double *z, const double *p, const double *Ap, const double *dinv, size_t n,
                    const double *rz, const double *pAp);
/* trilinear transfer between nested structured node lattices (coarse Nc, fine 2Nc-1 per axis), 3 dofs per node:
 * the h-multigrid that stands in for GAMG on the assembled p = 1 level (elasticity.c:569-585) */
int b200_lattice_prolong(int Ncx, int Ncy, int Ncz, const double *xc, double *xf);   /* xf = P xc   */
int b200_lattice_restrict(int Ncx, int Ncy, int Ncz, const double *xf, double *xc);  /* xc = P^T xf */
/* Chebyshev + point-Jacobi smoother (elasticity.c:539-552), fused vector updates:
 *   init: d = dinv .* r * inv_theta;  x = zero_guess ? d : x + d
 *   step: r -= Ad;  d = c1 d + c2 dinv .* r;  x += d */
int b200_cheb_init(double *x, const double *r, double *d, const double *dinv, double inv_theta, int zero_guess, size_t n);
int b200_cheb_step(double *x, double *r, double *d, const double *Ad, const double *dinv, double c1, double c2, size_t n);
/* assembled coarse operator on a structured (Nx,Ny,Nz) node lattice, 3 dofs per node, as a 27-point block
 * stencil: vals[((dx+1)+3(dy+1)+9(dz+1))*3 + a][row]; y = A x */
int b200_stencil27_spmv(int Nx, int Ny, int Nz, const double *vals, const double *x, double *y);
/* assembled coarse-level operator (FormJacobian by colouring, src/misc.c:151-183) in slot-major ELL:
 * y[r] = sum_s vals[s*n + r] * x[cols[s*n + r]]   (cols < 0 = empty slot) */
int b200_ell_spmv(size_t n, int nslots, const int *cols, const double *vals, const double *x, double *y);
/* `count` runs of `n` entries, `stride` apart, set to `value` */
int b200_fill_strided(double *d, double value, size_t n, size_t stride, size_t count);

/* ---- layout of CEED_STRIDES_BACKEND vectors (setuplibceed.c:304-318) --------------- */
/* The backend owns this layout.  For elemsize = Q^3 (2 <= Q <= 8) it is "q-blocked":
 * elements in groups of EB = b200_elems_per_block(Q); inside group g holding ebn
 * elements (ebn = EB except in the tail group), with q = qx + Q*t, t = qy + Q*qz:
 *   index(e,c,q) = g*EB*ncomp*Q^3 + (c*Q + qx)*(ebn*Q^2) + t*ebn + (e % EB)
 * i.e. [group][comp][qx][t][elem-in-group]: the fused kernels' lane id (t*ebn + e) walks
 * contiguous memory for every (comp, qx).  Otherwise plain [elem][comp][node]. */
int b200_elems_per_block(int Q);
int b200_strided_layout_q(int elemsize);  /* returns Q if the blocked layout applies, else 0 */

/* ---- generic path: CeedElemRestrictionApply (App. B.1) ----------------------------- */
/* offsets restriction: E[e][c][n] <-> L[offsets[e*elemsize+n] + c*compstride] */
int b200_restrict_offsets(int transpose, int nelem, int elemsize, int ncomp, int compstride,
                          const int *d_offsets, const double *d_in, double *d_out);
/* strided restriction; layout_q > 0 selects the q-blocked backend layout, else the three
 * strides {node, comp, elem} are used */
int b200_restrict_strided(int transpose, int nelem, int elemsize, int ncomp, int layout_q,
                          long long s_node, long long s_comp, long long s_elem,
                          const double *d_in, double *d_out);

/* ---- generic path: CeedBasisApply for tensor H1 bases, dim = 3 (App. B.3) ---------- */
/* emode: 1 INTERP, 2 GRAD, 4 WEIGHT.  E layout [elem][comp][P^3]; Q layouts
 * INTERP [elem][comp][Q^3], GRAD [elem][dim][comp][Q^3], WEIGHT [elem][Q^3].
 * d_interp1d/d_grad1d: device [Q*P]; d_qweight1d: device [Q]. */
int b200_basis_apply(int nelem, int ncomp, int P, int Q, const double *d_interp1d,
                     const double *d_grad1d, const double *d_qweight1d, int transpose, int emode,
                     const double *d_u, double *d_v);

/* ---- generic path: CeedQFunctionApply for recognised QFunctions (App. B.4) ---------- */
/* in[k] / out[k]: device Q-vectors [elem][size_k][nq] in field declaration order.
 * h_ctx: the QFunction context as HOST doubles ({nu, E} for the material models and the MMS forcing,
 * the 3-vector for the constant forcing; may be NULL when the QFunction takes none) */
int b200_qfunction_apply(int qf_id, const double *h_ctx, int nctx, int identity_size, int nelem, int nq,
                         int nin, const double *const *d_in, int nout, double *const *d_out);
/* the same point functions on the HOST (host Q-vectors, no GPU work): lets the backend compare the caller's own
 * QFunction pointer (setuplibceed.c:370-372,518-520,818-820) with its device body on a few known points */
int b200_qfunction_apply_host(int qf_id, const double *h_ctx, int nctx, int identity_size, int nelem, int nq,
                              int nin, const double *const *h_in, int nout, double *const *h_out);

/* generic-path piece of CeedOperatorLinearAssembleDiagonal (App. B.5): one unit-input pass,
 * ediag[e][cin][n] += sum_q sum_dout G_dout[q,n] dv[e][dout*3+cin][q] G_din[q,n]
 * (dv = QFunction output for the unit field (din, cin); G_d = Kronecker gradient matrices) */
int b200_diag_accumulate(int nelem, int P, int Q, const double *d_interp1d, const double *d_grad1d, int din,
                         int cin, const double *d_dv, double *d_ediag);

/* ---- hot path: fused CeedOperatorApply (matops.c:46; setuplibceed.c:518-542,818-839) */
/* y_L += E^T G^T D G E x_L in ONE kernel: offsets gather, sum-factorised gradient
 * (interpolate + collocated derivative), QFunction, transposed gradient, scatter-add.
 *   interp1d, grad1d : HOST [Q*P] basis matrices (CeedBasisCreateTensorH1Lagrange)
 *   qdata            : device, backend strided layout, 10 comps
 *   gradu            : device, backend strided layout, 9 comps (written; NULL for linElas)
 * Supported: 2 <= P <= Q <= 8 (P, Q as instantiated; see b200_fused_supported). */
int b200_fused_supported(int P, int Q);
/* shared-memory lattice of the fused apply kernel (tests: bank-conflict freedom): out[6] = {stride y, stride z,
 * component stride, element stride (all in doubles), elements per CTA, threads per CTA} */
int b200_apply_smem_layout(int P, int Q, int *out);
/* d_evec (all fused kernels): NULL = scatter-add with FP64 atomics straight into the L-vector.  Non-NULL selects
 * the DETERMINISTIC scatter: the kernel stores its element outputs to d_evec[(e*P^3 + node)*3 + comp] instead
 * (plain coalesced stores, d_y untouched) and the caller sums them into the L-vector in a fixed order with
 * b200_transpose_gather_add (layout 1).
 * Sub-ranges (residual, Jacobian, diagonal): d_offsets, d_qdata / d_gradu / d_jcache and d_evec may point at the
 * first element of a range that starts at a multiple of EB = b200_elems_per_block(Q).  nelem must then be a multiple
 * of EB unless the range runs to the end of the q-blocked vectors: the last group's extent is taken from nelem, and
 * the q-blocked layout of a group cut short would be that of the whole vector's group. */
int b200_apply_residual(int problem, const b200_physics *phys, int nelem, int P, int Q,
                        const double *h_interp1d, const double *h_grad1d, const int *d_offsets,
                        const double *d_qdata, double *d_gradu, const double *d_x, double *d_y, double *d_evec);

/* Ordered transpose of an offsets restriction (the serial scatter of /cpu/self, matops.c:46 -> CeedOperatorApply):
 *   L[o + c*compstride] += sum over the E-vector positions p = e*elemsize + n with offsets[p] == o, ASCENDING p
 * d_tptr [lsize+1], d_tidx [nelem*elemsize]: CSR of positions by offset value (b200_transpose_map_build).
 * layout 0: E[(e*ncomp + c)*elemsize + n] (libCEED E-vector);  layout 1: E[(e*elemsize + n)*ncomp + c]. */
int b200_transpose_gather_add(int lsize, const int *d_tptr, const int *d_tidx, int elemsize, int ncomp, int compstride,
                              int layout, const double *d_evec, double *d_L);
/* counting sort of the positions by offset on the HOST (set-up only): tptr [lsize+1], tidx [n] */
int b200_transpose_map_build(int lsize, size_t n, const int *h_offsets, int *h_tptr, int *h_tidx);

/* Jacobian cache ("jcache"): per quadrature point, everything the Jacobian action needs
 * in its cheapest algebraic form, built from (qdata, gradu) once per linearisation point
 * and shared by all p-multigrid levels (they share the fine quadrature data,
 * setuplibceed.c:757,833-839).  Components per problem: b200_jcache_ncomp(). */
int b200_jcache_ncomp(int problem);
int b200_jcache_build(int problem, int nelem, int Q, const double *d_qdata, const double *d_gradu,
                      double *d_jcache);
int b200_apply_jacobian(int problem, const b200_physics *phys, int nelem, int P, int Q,
                        const double *h_interp1d, const double *h_grad1d, const int *d_offsets,
                        const double *d_jcache, const double *d_x, double *d_y, double *d_evec);

/* CeedOperatorLinearAssembleDiagonal (matops.c:227; App. B.5): diag_L += E^T diag_e */
int b200_apply_diagonal(int problem, const b200_physics *phys, int nelem, int P, int Q,
                        const double *h_interp1d, const double *h_grad1d, const int *d_offsets,
                        const double *d_jcache, double *d_diag, double *d_evec);

/* ---- halo exchange over NVLink peer memory (one node, one process per GPU; the DMLocalToGlobal(ADD) +
 * DMGlobalToLocal(INSERT) pair of matops.c:33,57 as one symmetric sum-and-share, no communication library on the
 * data path).  Each rank owns a window of b200_halo_window_bytes(total) bytes
 *     [parity 0: total doubles | parity 1: total doubles | one int64 flag per neighbour | generation | error word]
 * allocated with b200_malloc (zeroed) and exported with CUDA IPC; neighbours store their partial sums into it.
 *   b200_halo_begin  (side stream, high priority, ordered behind everything queued on the compute stream): packed
 *                    position i of segment s (seg_start[s] <= i < seg_start[s+1]) of d_y[d_idx[i]] is stored to
 *                    remote_p{parity}[s][i - seg_start[s]], then *remote_flag[s] = generation (release, system scope);
 *   b200_halo_end    (compute stream): waits until every neighbour's flag shows this generation (bounded by timeout_s;
 *                    on expiry the error word is set and the kernel returns -- loud failure instead of a hung GPU), then
 *                    for every unique shared dof u: y[udof[u]] = sum over uent[uptr[u] .. uptr[u+1]) in that order of
 *                    (entry < 0 ? y[udof[u]] : window[entry]) -- the holders' partial sums in ascending rank order, so
 *                    every holder computes the bit-identical total, without atomics.
 * The caller may keep the compute stream busy between begin and end with work that does not touch shared dofs. */
#define B200_HALO_MAX_NEIGHBOURS 32
typedef struct b200_halo b200_halo;
int b200_ipc_get_handle(const void *dptr, unsigned char *handle64);
int b200_ipc_open(const unsigned char *handle64, void **dptr);
int b200_ipc_close(void *dptr);
size_t b200_halo_window_bytes(size_t total);
int b200_halo_create(int nnbr, const int *seg_start, double *const *remote_p0, double *const *remote_p1,
                     long long *const *remote_flag, const int *d_idx, size_t total, void *d_window, int nuniq,
                     const int *d_udof, const int *d_uptr, const int *d_uent, double timeout_s, b200_halo **out);
int b200_halo_destroy(b200_halo *h);
int b200_halo_begin(b200_halo *h, const double *d_y);
/* fork/begin_forked: the work that produces the interface partial sums is queued on the halo's side stream
 * (b200_halo_fork orders it behind the compute stream and returns it; the caller switches b200_set_stream to it and
 * back), so it runs CONCURRENTLY with shared-dof-free work on the compute stream; the push follows it on the side stream */
int b200_halo_fork(b200_halo *h, void **side_stream);
int b200_halo_begin_forked(b200_halo *h, const double *d_y);
int b200_halo_end(b200_halo *h, double *d_y);
int b200_halo_error(b200_halo *h, int *err);   /* synchronises; *err != 0: an exchange timed out */
/* the same ordered sum for exchanges carried by a communication library (d_recv laid out like a window) */
int b200_halo_unpack_ordered(int nuniq, const int *d_udof, const int *d_uptr, const int *d_uent, const double *d_recv,
                             double *d_y);

/* FP64 pipe probe: sustained DFMA/s of the device (8 independent chains per thread), for the FP64 cross-check of the
 * HBM roofline (SURVEY.md 8(d)); synchronises */
int b200_fp64_probe(double *dfma_per_second);

/* Host-resident L-vectors (-memtype host; CeedVectorSetArray(HOST) ... TakeArray(HOST), matops.c:40-50): the fused
 * apply as a pipeline  H2D of x chunks | kernel on element chunks | D2H of finished y rows  on three streams.
 * chunk_end[c] = one past the last element of chunk c (multiples of b200_elems_per_block(Q) except the last);
 * in_need[c]   = length of the x prefix chunk c reads;  out_final[c] = length of the y prefix no later chunk touches.
 * d_y must already be zeroed on the compute stream; h_x, h_y page-locked (b200_host_is_pinned).  Synchronous. */
int b200_host_is_pinned(const void *p);
int b200_apply_hostpipe(int jacobian, int problem, const b200_physics *phys, int nelem, int P, int Q,
                        const double *h_interp1d, const double *h_grad1d, const int *d_offsets, const double *d_qa,
                        double *d_gradu, const double *h_x, double *d_x, double *h_y, double *d_y, size_t lsize,
                        int nchunks, const int *chunk_end, const size_t *in_need, const size_t *out_final);

/* CeedOperatorLinearAssemble for a trilinear (P = 2) Jacobian level: element matrices straight from the Jacobian
 * cache, d_values[(e*24 + col)*24 + row], element dof = node*3 + component (node = ix + 2 iy + 4 iz).  Replaces
 * the 81 coloured operator applications of FormJacobian (misc.c:151-183) by one pass over the cache. */
int b200_assemble_p1(int problem, const b200_physics *phys, int nelem, int Q, const double *h_interp1d,
                     const double *h_grad1d, const double *d_jcache, double *d_values);

/* Galerkin product A_H = P^T A_h P of 27-point block stencils (layout of b200_stencil27_spmv) on 2:1 nested
 * node lattices, fine lattice 2*Nc - 1 per axis, trilinear index-space P (b200_lattice_prolong) */
int b200_stencil27_galerkin(int Ncx, int Ncy, int Ncz, const double *d_fine, double *d_coarse);

/* p-multigrid transfer (matops.c:115-203): out_L += Eo^T I^(T) Ei in_L, identity QFunction,
 * interpolation Pc -> Pf at the fine GLL points; transpose = 1 is the restriction.
 * d_mult (may be NULL): fine-level inverse multiplicity applied to the fine vector
 * (after prolongation / before restriction, matops.c:149,176).
 * inject (prolongation with d_mult only): out_L[fine node] = interpolant, stored instead of summed and scaled --
 * the elements sharing a fine node all interpolate the same value there (continuous coarse field), so
 * sum x 1/multiplicity is that value; no atomics, no pre-zeroed output, no read of d_mult.  Bit for bit only
 * where the sharing elements have the same local axes: a differently oriented one contracts in another order. */
int b200_apply_transfer(int transpose, int nelem, int Pc, int Pf, const double *h_interpCtoF,
                        const int *d_offc, const int *d_offf, const double *d_mult, int inject,
                        const double *d_in, double *d_out, double *d_evec);

/* ---- smoothed-aggregation AMG on the assembled p = 1 level (the GAMG coarse solve, elasticity.c:569-585) -------
 * BSR matrices: block rows rowptr[nbrows+1], block columns colidx[nnzb], values [nnzb][br][bc] (row-major blocks).
 * Every output is a fixed-order sum of its listed terms (no atomics): results are bit-identical from run to run. */
/* y = A x; block shapes (br, bc) in {(3,3), (6,6), (3,6), (6,3)} */
int b200_bsr_spmv(int br, int bc, int nbrows, const int *rowptr, const int *colidx, const double *vals,
                  const double *x, double *y);
/* pair-list block product C[k] = sum_{t = ptr[k]}^{ptr[k+1]-1} A[pa[t]] B[pb[t]]  (br x bk times bk x bc blocks);
 * (br, bk, bc) in {(3,3,6), (6,3,6), (6,6,6), (3,3,3)}.  tmap != NULL selects the smoothed-prolongator epilogue
 *   C[k] = T[tmap[k]] - omega[0] * dinv[rowof[k]*br + i] * C[k]   (row i of the block; tmap[k] < 0: T block absent)
 * with omega a DEVICE scalar (no host synchronisation) */
int b200_bsr_pairs_product(int br, int bk, int bc, size_t nout, const long long *ptr, const int *pa, const int *pb,
                           const double *A, const double *B, double *C, const int *tmap, const int *rowof,
                           const double *T, const double *dinv, const double *omega);
/* dst[k] = src[idx[k]]^T (src blocks br x bc, dst blocks bc x br): the transposed prolongator by a fixed gather;
 * (br, bc) in {(3,6), (6,6), (3,3)} */
int b200_bsr_transpose_gather(int br, int bc, size_t nblocks, const int *idx, const double *src, double *dst);
/* 3x3 blocks from element matrices evals[(e*24 + col)*24 + row] (b200_assemble_p1 layout):
 *   vals[k][i][j] = sum_{t = ptr[k]}^{ptr[k+1]-1} evals[src[t] + 24 j + i]   (src[t] = (e*24 + 3b)*24 + 3a) */
int b200_bsr_assemble_elem(size_t nblocks, const long long *ptr, const long long *src, const double *evals,
                           double *vals);

/* ---- K11: user QFunctions compiled at run time with NVRTC ("/gpu/b200:jit", csrc/b200_jit.cu) ---------------------
 * b200_jit_read_source (host only): the program text of the QFunction source file `path` (used as given), every quoted
 *   #include "..." that exists next to its includer inlined recursively between #line directives.  *text: free with
 *   b200_jit_free_source.  On failure returns != 0 with the reason (naming the path) in err.
 * b200_jit_compile (no device needed): text + the generated kernel for QFunction `name` with the given field sizes
 *   (Q-vectors [elem][size][nq]), compiled by NVRTC for sm_100a unless the same program was compiled before in this
 *   process; *handle names it.  Errors carry the NVRTC log (about 4 KB at most) in b200_last_error().
 * b200_jit_apply: one launch on the backend stream; the context (at most B200_JIT_MAX_CTX bytes) is copied from the
 *   host pointer at every call.  The user function's return code is ignored.
 * b200_jit_compile_count: NVRTC compilations run by this process.  b200_jit_program: the compiled program text. */
#define B200_JIT_MAX_CTX 2048
#define B200_JIT_MAX_FIELD 64
#define B200_JIT_MAXF 8
int b200_jit_read_source(const char *path, char **text, char *err, size_t errlen);
void b200_jit_free_source(char *text);
int b200_jit_compile(const char *text, const char *src_name, const char *name, int nin, const int *in_sizes, int nout,
                     const int *out_sizes, int *handle);
int b200_jit_apply(int handle, const void *h_ctx, size_t ctx_bytes, int nelem, int nq, int nin, const double *const *d_in,
                   int nout, double *const *d_out);
unsigned long long b200_jit_compile_count(void);
const char *b200_jit_program(int handle);

/* ---- K12: the fused operator kernel around a JIT-compiled user QFunction (csrc/b200_jit_fused.cuh) ----------------
 * b200_jit_fused_compile (no device needed): text + the kernel of b200_jit_fused.cuh around QFunction `name` for the
 *   basis (P, Q) (one of b200_fused_supported; the lattice constants are those of b200_apply_smem_layout).  Field
 *   active_in is the 9-component gradient of the 3-component offsets-restricted active vector, in[d*3 + c] = du_c/dX_d;
 *   field active_out is its 9-component test-function gradient, out[k*3 + c].  Every other field is a passive vector
 *   in the q-blocked CEED_STRIDES_BACKEND layout, read (inputs) or written (outputs) in place.  Compiled unless the
 *   same program (text, name, sizes, active fields, P, Q) was compiled before; counted by b200_jit_compile_count and
 *   shown by b200_jit_program.
 * b200_jit_fused_apply: y_L += E^T G^T f(G E x_L, passive fields) G E on nelem elements, one launch for the full
 *   element groups and one for a partial last group, on the backend stream.  d_offsets, d_in / d_out of the passive
 *   fields and d_evec point at the first element of the range (a multiple of b200_elems_per_block(Q)); nelem is a
 *   multiple of it too unless the range runs to the end of the q-blocked passive vectors (as for the built-in fused
 *   kernels above); entries of the active fields are ignored.  passive_add = 0 stores the passive outputs, != 0 adds to them.  d_evec as for the
 *   built-in fused kernels (NULL: FP64 atomics; else E-vector [e][node][comp] for b200_transpose_gather_add).  The
 *   context is copied from the host pointer at every call (at most B200_JIT_MAX_CTX bytes). */
int b200_jit_fused_compile(const char *text, const char *src_name, const char *name, int nin, const int *in_sizes,
                           int nout, const int *out_sizes, int active_in, int active_out, int P, int Q, int *handle);
int b200_jit_fused_apply(int handle, const void *h_ctx, size_t ctx_bytes, int nelem, const double *h_interp1d,
                         const double *h_grad1d, const int *d_offsets, const double *d_x, double *d_y, double *d_evec,
                         int nin, const double *const *d_in, int nout, double *const *d_out, int passive_add);

/* ---- K13: element matrices of a trilinear level around a JIT-compiled user QFunction (csrc/b200_jit_assemble.cuh) --
 * b200_jit_assemble_compile (no device needed): text + the kernel of b200_jit_assemble.cuh around QFunction `name`
 *   for the basis (P, Q) = (2, Q), Q one of B200_FOR_PQ; fields as for b200_jit_fused_compile.  Any other P, or an
 *   active field that is not 9 wide, is refused.  Compiled unless the same program (text, name, sizes, active fields,
 *   Q) was compiled before; counted by b200_jit_compile_count and shown by b200_jit_program.
 * b200_jit_assemble_apply: the CeedOperatorLinearAssemble values of nelem elements, layout of b200_assemble_p1:
 *   d_values[(e*24 + col)*24 + row] = sum_q G_row(q)^T D_q G_col(q), D_q the point tangent of the user function,
 *   dout_active / din_active, from its 9 calls with the unit active inputs at point q (passive inputs as given, passive
 *   outputs discarded; the return code is ignored).  This is the Jacobian only if the function is linear in its
 *   active input.  One launch for the full element groups and one for a partial last group, on the backend stream;
 *   no atomics (bit-identical from run to run).  d_in of the passive inputs: q-blocked vectors of nelem elements;
 *   entries of the active field are ignored.  The context is copied from the host pointer at every call (at most
 *   B200_JIT_MAX_CTX bytes). */
int b200_jit_assemble_compile(const char *text, const char *src_name, const char *name, int nin, const int *in_sizes,
                              int nout, const int *out_sizes, int active_in, int active_out, int P, int Q, int *handle);
int b200_jit_assemble_apply(int handle, const void *h_ctx, size_t ctx_bytes, int nelem, const double *h_interp1d,
                            const double *h_grad1d, int nin, const double *const *d_in, double *d_values);

/* ---- K14: the operator diagonal around a JIT-compiled user QFunction (csrc/b200_jit_diag.cuh) ----------------------
 * b200_jit_diag_compile (no device needed): text + the kernel of b200_jit_diag.cuh around QFunction `name` for the
 *   basis (P, Q) (one of b200_fused_supported; the lattice constants are those of b200_apply_smem_layout); fields as
 *   for b200_jit_fused_compile.  Any other (P, Q), or an active field that is not 9 wide, is refused.  Compiled unless
 *   the same program (text, name, sizes, active fields, P, Q) was compiled before; counted by b200_jit_compile_count
 *   and shown by b200_jit_program.
 * b200_jit_diag_apply: d_diag += the diagonal of E^T G^T D_q G E on nelem elements, D_q the point tangent of the user
 *   function, dout_active / din_active, from 3 calls per point and component with the unit active inputs (passive
 *   inputs as given, passive outputs discarded; the return code is ignored).  The off-diagonal gradient terms enter as
 *   D[c d][c d'] + D[c d'][c d], so a non-symmetric tangent is handled.  This is the operator's diagonal only if the
 *   function is linear in its active input.  One launch for the full element groups and one for a partial last group,
 *   on the backend stream.  d_evec NULL: FP64 atomics into d_diag at d_offsets + c; else d_evec [e][node][comp] is
 *   stored for b200_transpose_gather_add and d_diag is untouched.  d_in of the passive inputs: q-blocked vectors of
 *   nelem elements; entries of the active field are ignored.  The context is copied from the host pointer at every
 *   call (at most B200_JIT_MAX_CTX bytes). */
int b200_jit_diag_compile(const char *text, const char *src_name, const char *name, int nin, const int *in_sizes,
                          int nout, const int *out_sizes, int active_in, int active_out, int P, int Q, int *handle);
int b200_jit_diag_apply(int handle, const void *h_ctx, size_t ctx_bytes, int nelem, const double *h_interp1d,
                        const double *h_grad1d, const int *d_offsets, int nin, const double *const *d_in,
                        double *d_diag, double *d_evec);

#ifdef __cplusplus
}
#endif
#endif /* B200_KERNELS_H */
