// Smoothed-aggregation AMG coarse solve on the assembled p = 1 level (the GAMG stand-in for unstructured meshes,
// elasticity.c:569-585): block-sparse (BSR) mat-vec, pair-list block products for the Galerkin set-up, the
// transposed prolongator by a fixed gather, and the level-0 BSR matrix from the element matrices.
// Every output is a fixed-order sum of its listed terms: no atomics, bit-identical from run to run.
#include "b200_common.cuh"

namespace b200 {
namespace {

inline int grid_for(size_t n, int nt) {
  size_t g = (n + nt - 1) / nt;
  return (int)(g < 1 ? 1 : (g > 1048576 ? 1048576 : g));
}

// y = A x, BSR with BR x BC blocks (row-major inside a block), one warp per block row.  The values of a block row
// are contiguous, so the warp streams them with unit stride (lane l reads entries l, l+32, ...); each lane keeps one
// partial sum per block-row component and the warp reduces them by shuffles at the end.
template <int BR, int BC>
__global__ void k_bsr_spmv(int nbrows, const int *__restrict__ rowptr, const int *__restrict__ colidx,
                           const double *__restrict__ vals, const double *__restrict__ x, double *__restrict__ y) {
  constexpr int BB = BR * BC;
  const int lane = threadIdx.x & 31;
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < nbrows; row += warps) {
    const int b0 = rowptr[row], b1 = rowptr[row + 1];
    const size_t e0 = (size_t)b0 * BB, e1 = (size_t)b1 * BB;
    double acc[BR];
#pragma unroll
    for (int i = 0; i < BR; i++) acc[i] = 0.0;
    for (size_t e = e0 + lane; e < e1; e += 32) {
      const size_t blk = e / BB;
      const int w = (int)(e - blk * BB), i = w / BC, j = w - i * BC;
      const double prod = vals[e] * x[(size_t)colidx[blk] * BC + j];
#pragma unroll
      for (int r = 0; r < BR; r++) acc[r] += (i == r) ? prod : 0.0;
    }
#pragma unroll
    for (int r = 0; r < BR; r++) {
      double v = acc[r];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      acc[r] = v;
    }
    if (lane < BR) {
      double v = acc[0];
#pragma unroll
      for (int r = 1; r < BR; r++) v = (lane == r) ? acc[r] : v;
      y[(size_t)row * BR + lane] = v;
    }
  }
}

// C[k] = sum_{t = ptr[k]}^{ptr[k+1]-1} A[pa[t]] B[pb[t]]  (BR x BK times BK x BC blocks), in list order; one thread
// per output entry (k, i, j).  Epilogue (tmap != NULL), the smoothed prolongator:
//   C[k] = T[tmap[k]] - omega dinv[rowof[k]*BR + i] C[k]   (tmap[k] < 0: no tentative block there)
template <int BR, int BK, int BC>
__global__ void k_bsr_pairs(size_t nout, const long long *__restrict__ ptr, const int *__restrict__ pa,
                            const int *__restrict__ pb, const double *__restrict__ A, const double *__restrict__ B,
                            double *__restrict__ C, const int *__restrict__ tmap, const int *__restrict__ rowof,
                            const double *__restrict__ T, const double *__restrict__ dinv,
                            const double *__restrict__ omega) {
  constexpr int BB = BR * BC;
  for (size_t g = blockIdx.x * (size_t)blockDim.x + threadIdx.x; g < nout * BB; g += (size_t)gridDim.x * blockDim.x) {
    const size_t k = g / BB;
    const int w = (int)(g - k * BB), i = w / BC, j = w - i * BC;
    double s = 0.0;
    for (long long t = ptr[k]; t < ptr[k + 1]; t++) {
      const double *a = A + (size_t)pa[t] * (BR * BK) + i * BK;
      const double *b = B + (size_t)pb[t] * (BK * BC) + j;
#pragma unroll
      for (int m = 0; m < BK; m++) s += a[m] * b[m * BC];
    }
    if (tmap != nullptr) {
      const int tk = tmap[k];
      const double t0 = tk >= 0 ? T[(size_t)tk * BB + w] : 0.0;
      s = t0 - omega[0] * dinv[(size_t)rowof[k] * BR + i] * s;
    }
    C[g] = s;
  }
}

// dst[k] = src[idx[k]]^T  (src blocks BR x BC, dst blocks BC x BR)
template <int BR, int BC>
__global__ void k_bsr_transpose_gather(size_t nblocks, const int *__restrict__ idx, const double *__restrict__ src,
                                       double *__restrict__ dst) {
  constexpr int BB = BR * BC;
  for (size_t g = blockIdx.x * (size_t)blockDim.x + threadIdx.x; g < nblocks * BB;
       g += (size_t)gridDim.x * blockDim.x) {
    const size_t k = g / BB;
    const int w = (int)(g - k * BB), i = w / BR, j = w - i * BR;  // dst entry (i, j) = src entry (j, i)
    dst[g] = src[(size_t)idx[k] * BB + j * BC + i];
  }
}

// level-0 3x3 blocks from element matrices E[(e*24 + col)*24 + row]: block k, entry (i, j) =
// sum_{t = ptr[k]}^{ptr[k+1]-1} E[src[t] + 24 j + i], in list order
__global__ void k_bsr_assemble_elem(size_t nblocks, const long long *__restrict__ ptr, const long long *__restrict__ src,
                                    const double *__restrict__ E, double *__restrict__ vals) {
  for (size_t g = blockIdx.x * (size_t)blockDim.x + threadIdx.x; g < nblocks * 9; g += (size_t)gridDim.x * blockDim.x) {
    const size_t k = g / 9;
    const int w = (int)(g - k * 9), i = w / 3, j = w - i * 3;
    double s = 0.0;
    for (long long t = ptr[k]; t < ptr[k + 1]; t++) s += E[src[t] + 24 * j + i];
    vals[g] = s;
  }
}

template <int BR, int BC>
int launch_spmv(int nbrows, const int *rowptr, const int *colidx, const double *vals, const double *x, double *y) {
  if (nbrows <= 0) return 0;
  const int nt = 256;
  k_bsr_spmv<BR, BC><<<grid_for((size_t)nbrows * 32, nt), nt, 0, g_stream>>>(nbrows, rowptr, colidx, vals, x, y);
  B200_LAUNCH_CHECK("k_bsr_spmv");
  return 0;
}

template <int BR, int BK, int BC>
int launch_pairs(size_t nout, const long long *ptr, const int *pa, const int *pb, const double *A, const double *B,
                 double *C, const int *tmap, const int *rowof, const double *T, const double *dinv,
                 const double *omega) {
  if (nout == 0) return 0;
  const int nt = 128;
  k_bsr_pairs<BR, BK, BC><<<grid_for(nout * BR * BC, nt), nt, 0, g_stream>>>(nout, ptr, pa, pb, A, B, C, tmap, rowof, T,
                                                                              dinv, omega);
  B200_LAUNCH_CHECK("k_bsr_pairs");
  return 0;
}

template <int BR, int BC>
int launch_tgather(size_t nblocks, const int *idx, const double *src, double *dst) {
  if (nblocks == 0) return 0;
  k_bsr_transpose_gather<BR, BC><<<grid_for(nblocks * BR * BC, 256), 256, 0, g_stream>>>(nblocks, idx, src, dst);
  B200_LAUNCH_CHECK("k_bsr_transpose_gather");
  return 0;
}

}  // namespace
}  // namespace b200

using namespace b200;

extern "C" {

int b200_bsr_spmv(int br, int bc, int nbrows, const int *rowptr, const int *colidx, const double *vals,
                  const double *x, double *y) {
  if (br == 3 && bc == 3) return launch_spmv<3, 3>(nbrows, rowptr, colidx, vals, x, y);
  if (br == 6 && bc == 6) return launch_spmv<6, 6>(nbrows, rowptr, colidx, vals, x, y);
  if (br == 3 && bc == 6) return launch_spmv<3, 6>(nbrows, rowptr, colidx, vals, x, y);
  if (br == 6 && bc == 3) return launch_spmv<6, 3>(nbrows, rowptr, colidx, vals, x, y);
  return set_error_msg("b200_bsr_spmv: block shape not instantiated (3x3, 6x6, 3x6, 6x3)");
}

int b200_bsr_pairs_product(int br, int bk, int bc, size_t nout, const long long *ptr, const int *pa, const int *pb,
                           const double *A, const double *B, double *C, const int *tmap, const int *rowof,
                           const double *T, const double *dinv, const double *omega) {
  if (tmap != nullptr && (rowof == nullptr || dinv == nullptr || omega == nullptr))
    return set_error_msg("b200_bsr_pairs_product: the epilogue needs rowof, dinv and omega");
  if (br == 3 && bk == 3 && bc == 6) return launch_pairs<3, 3, 6>(nout, ptr, pa, pb, A, B, C, tmap, rowof, T, dinv, omega);
  if (br == 6 && bk == 3 && bc == 6) return launch_pairs<6, 3, 6>(nout, ptr, pa, pb, A, B, C, tmap, rowof, T, dinv, omega);
  if (br == 6 && bk == 6 && bc == 6) return launch_pairs<6, 6, 6>(nout, ptr, pa, pb, A, B, C, tmap, rowof, T, dinv, omega);
  if (br == 3 && bk == 3 && bc == 3) return launch_pairs<3, 3, 3>(nout, ptr, pa, pb, A, B, C, tmap, rowof, T, dinv, omega);
  return set_error_msg("b200_bsr_pairs_product: block shape not instantiated (3x3*3x6, 6x3*3x6, 6x6*6x6, 3x3*3x3)");
}

int b200_bsr_transpose_gather(int br, int bc, size_t nblocks, const int *idx, const double *src, double *dst) {
  if (br == 3 && bc == 6) return launch_tgather<3, 6>(nblocks, idx, src, dst);
  if (br == 6 && bc == 6) return launch_tgather<6, 6>(nblocks, idx, src, dst);
  if (br == 3 && bc == 3) return launch_tgather<3, 3>(nblocks, idx, src, dst);
  return set_error_msg("b200_bsr_transpose_gather: block shape not instantiated (3x6, 6x6, 3x3)");
}

int b200_bsr_assemble_elem(size_t nblocks, const long long *ptr, const long long *src, const double *evals,
                           double *vals) {
  if (nblocks == 0) return 0;
  k_bsr_assemble_elem<<<grid_for(nblocks * 9, 256), 256, 0, g_stream>>>(nblocks, ptr, src, evals, vals);
  B200_LAUNCH_CHECK("k_bsr_assemble_elem");
  return 0;
}

}  // extern "C"
