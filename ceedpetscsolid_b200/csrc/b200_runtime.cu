// Runtime pieces of the thin C-ABI CUDA layer: device/stream/memory management,
// CeedVector kernels, index gather/scatter for the global<->local maps and halos.
#include <string.h>

#include "b200_common.cuh"

namespace b200 {
cudaStream_t g_stream = 0;
unsigned long long g_launches = 0;
static char g_err[8192] = "";  // room for an NVRTC log (b200_jit.cu)

int set_error(cudaError_t e, const char *what) {
  snprintf(g_err, sizeof g_err, "CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
  return (int)e;
}
int set_error_msg(const char *msg) {
  snprintf(g_err, sizeof g_err, "%s", msg);
  return 999;
}

static inline int grid_for(size_t n, int nt) {
  size_t nb = (n + nt - 1) / nt;
  const size_t cap = 148 * 32;
  return (int)(nb > cap ? cap : (nb ? nb : 1));
}

#define GRID_STRIDE(i, n) \
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < (n); i += (size_t)gridDim.x * blockDim.x)

__global__ void k_set(double *d, double v, size_t n) { GRID_STRIDE(i, n) d[i] = v; }
__global__ void k_recip(double *d, size_t n) {
  GRID_STRIDE(i, n) { const double v = d[i]; d[i] = fabs(v) > 1e-14 ? 1.0 / v : v; }  // CeedVectorReciprocal guards tiny entries
}
__global__ void k_scale(double *d, double a, size_t n) { GRID_STRIDE(i, n) d[i] *= a; }
__global__ void k_axpy(double *y, double a, const double *x, size_t n) { GRID_STRIDE(i, n) y[i] += a * x[i]; }
__global__ void k_aypx(double *y, double a, const double *x, size_t n) { GRID_STRIDE(i, n) y[i] = x[i] + a * y[i]; }
__global__ void k_axpby(double *z, double a, const double *x, double b, const double *y, size_t n) {
  GRID_STRIDE(i, n) z[i] = a * x[i] + b * y[i];
}
__global__ void k_pmult(double *w, const double *x, const double *y, size_t n) { GRID_STRIDE(i, n) w[i] = x[i] * y[i]; }
__global__ void k_gather(double *dst, const double *src, const int *idx, size_t n) { GRID_STRIDE(i, n) dst[i] = src[idx[i]]; }
__global__ void k_scatter_set(double *dst, const int *idx, const double *src, size_t n) { GRID_STRIDE(i, n) dst[idx[i]] = src[i]; }
__global__ void k_scatter_add(double *dst, const int *idx, const double *src, size_t n) {
  GRID_STRIDE(i, n) atomicAdd(dst + idx[i], src[i]);
}
__global__ void k_gather_or_zero(double *dst, const double *src, const int *idx, size_t n) {
  GRID_STRIDE(i, n) { const int j = idx[i]; dst[i] = j >= 0 ? src[j] : 0.0; }
}
__global__ void k_copy_where(double *dst, const double *src, const int *idx, size_t n) {
  GRID_STRIDE(i, n) { const int j = idx[i]; if (j >= 0) dst[i] = src[j]; }
}
// BLAS-1 with DEVICE scalars (alpha = sign * num[0] / den[0]): lets a Krylov loop run without host syncs
// num / den of two device-resident scalars of a sync-free Krylov loop.  When the iteration has converged exactly
// (r = 0 -> rz = 0, p = 0, pAp = 0) or broken down, the quotient would be 0/0: the step is then 0, so x, r and p
// freeze instead of turning into NaN (the loop looks at the residual only every few iterations).
__device__ __forceinline__ double guarded_ratio(double num, double den) {
  const double a = num / den;
  return (den != 0.0 && isfinite(a)) ? a : 0.0;
}
__global__ void k_axpy_dev(double *y, const double *x, size_t n, const double *num, const double *den, double sign) {
  const double a = sign * guarded_ratio(num[0], den[0]);
  GRID_STRIDE(i, n) y[i] += a * x[i];
}
__global__ void k_aypx_dev(double *y, const double *x, size_t n, const double *num, const double *den) {
  const double a = guarded_ratio(num[0], den[0]);
  GRID_STRIDE(i, n) y[i] = x[i] + a * y[i];
}
// CG update in one pass: x += alpha p, r -= alpha Ap, z = dinv .* r   (alpha = rz / pAp, device scalars)
__global__ void k_pcg_update(double *x, double *r, double *z, const double *p, const double *Ap, const double *dinv,
                             size_t n, const double *rz, const double *pAp) {
  const double a = guarded_ratio(rz[0], pAp[0]);
  GRID_STRIDE(i, n) {
    if (x) x[i] += a * p[i];  // x == NULL: Lanczos run for eigenvalue estimates, the iterate is not needed
    const double ri = r[i] - a * Ap[i];
    r[i] = ri;
    z[i] = dinv[i] * ri;
  }
}
// Chebyshev/Jacobi smoother, fused vector updates (one pass each instead of 3-4 BLAS-1 passes)
//   init: d = dinv .* r * inv_theta;  x = zero_guess ? d : x + d
//   step: r -= Ad;  d = c1 d + c2 dinv .* r;  x += d
__global__ void k_cheb_init(double *x, const double *r, double *d, const double *dinv, double inv_theta, int zero_guess,
                            size_t n) {
  GRID_STRIDE(i, n) {
    const double di = dinv[i] * r[i] * inv_theta;
    d[i] = di;
    x[i] = zero_guess ? di : x[i] + di;
  }
}
__global__ void k_cheb_step(double *x, double *r, double *d, const double *Ad, const double *dinv, double c1, double c2,
                            size_t n) {
  GRID_STRIDE(i, n) {
    const double ri = r[i] - Ad[i];
    const double di = c1 * d[i] + c2 * (dinv[i] * ri);
    r[i] = ri;
    d[i] = di;
    x[i] += di;
  }
}
// Trilinear transfer between nested structured node lattices (coarse Nc -> fine 2Nc-1 per axis), 3 dofs per node.
// prolong: xf = P xc;   restrict: xc = P^T xf   (gather form: each output entry is written by one thread)
__global__ void k_lattice_prolong(int Ncx, int Ncy, int Ncz, const double *__restrict__ xc, double *__restrict__ xf) {
  const int Nfx = 2 * Ncx - 1, Nfy = 2 * Ncy - 1, Nfz = 2 * Ncz - 1;
  const size_t n = (size_t)3 * Nfx * Nfy * Nfz;
  GRID_STRIDE(row, n) {
    const int a = (int)(row % 3), node = (int)(row / 3);
    const int i = node % Nfx, j = (node / Nfx) % Nfy, k = node / (Nfx * Nfy);
    const int i0 = i >> 1, j0 = j >> 1, k0 = k >> 1, di = i & 1, dj = j & 1, dk = k & 1;
    double s = 0;
    for (int c = 0; c <= dk; c++)
      for (int b = 0; b <= dj; b++)
        for (int e = 0; e <= di; e++) s += xc[(size_t)3 * ((i0 + e) + Ncx * ((j0 + b) + (size_t)Ncy * (k0 + c))) + a];
    xf[row] = s * (di ? 0.5 : 1.0) * (dj ? 0.5 : 1.0) * (dk ? 0.5 : 1.0);
  }
}
__global__ void k_lattice_restrict(int Ncx, int Ncy, int Ncz, const double *__restrict__ xf, double *__restrict__ xc) {
  const int Nfx = 2 * Ncx - 1, Nfy = 2 * Ncy - 1, Nfz = 2 * Ncz - 1;
  const size_t n = (size_t)3 * Ncx * Ncy * Ncz;
  GRID_STRIDE(row, n) {
    const int a = (int)(row % 3), node = (int)(row / 3);
    const int I = node % Ncx, J = (node / Ncx) % Ncy, K = node / (Ncx * Ncy);
    double s = 0;
    for (int dk = -1; dk <= 1; dk++) {
      const int k = 2 * K + dk;
      if (k < 0 || k >= Nfz) continue;
      for (int dj = -1; dj <= 1; dj++) {
        const int j = 2 * J + dj;
        if (j < 0 || j >= Nfy) continue;
        for (int di = -1; di <= 1; di++) {
          const int i = 2 * I + di;
          if (i < 0 || i >= Nfx) continue;
          const double w = (di ? 0.5 : 1.0) * (dj ? 0.5 : 1.0) * (dk ? 0.5 : 1.0);
          s += w * xf[(size_t)3 * (i + Nfx * (j + (size_t)Nfy * k)) + a];
        }
      }
    }
    xc[row] = s;
  }
}
// 27-point vector stencil on a structured node lattice: vals[(o*3 + a)*n + row], o = (dx+1)+3(dy+1)+9(dz+1)
__global__ void k_stencil27_spmv(int Nx, int Ny, int Nz, const double *__restrict__ vals, const double *__restrict__ x,
                                 double *__restrict__ y) {
  const size_t n = (size_t)3 * Nx * Ny * Nz;
  GRID_STRIDE(row, n) {
    const int node = (int)(row / 3);
    const int i = node % Nx, j = (node / Nx) % Ny, k = node / (Nx * Ny);
    double s = 0;
    for (int dz = -1; dz <= 1; dz++) {
      if (k + dz < 0 || k + dz >= Nz) continue;
      for (int dy = -1; dy <= 1; dy++) {
        if (j + dy < 0 || j + dy >= Ny) continue;
        for (int dx = -1; dx <= 1; dx++) {
          if (i + dx < 0 || i + dx >= Nx) continue;
          const int o = (dx + 1) + 3 * (dy + 1) + 9 * (dz + 1);
          const size_t col = (size_t)3 * (node + dx + Nx * (dy + Ny * dz));
#pragma unroll
          for (int a = 0; a < 3; a++) s += vals[(size_t)(o * 3 + a) * n + row] * x[col + a];
        }
      }
    }
    y[row] = s;
  }
}
// ELL sparse mat-vec (slot-major storage): y[r] = sum_s vals[s*n + r] * x[cols[s*n + r]], cols < 0 = empty
__global__ void k_ell_spmv(size_t n, int nslots, const int *__restrict__ cols, const double *__restrict__ vals,
                           const double *__restrict__ x, double *__restrict__ y) {
  GRID_STRIDE(r, n) {
    double s = 0;
    for (int k = 0; k < nslots; k++) {
      const int c = cols[(size_t)k * n + r];
      if (c >= 0) s += vals[(size_t)k * n + r] * x[c];
    }
    y[r] = s;
  }
}
__global__ void k_fp64_probe(double *sink, int iters, double m) {
  double a0 = threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
  const double c = 1e-9;
#pragma unroll 4
  for (int i = 0; i < iters; i++) {
    a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
    a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
  }
  sink[blockIdx.x * (size_t)blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}
__global__ void k_fill_strided(double *d, double v, size_t n, size_t stride, size_t count) {
  GRID_STRIDE(i, n * count) d[(i / n) * stride + i % n] = v;
}
__global__ void k_mask_zero(double *d, const int *idx, size_t n) { GRID_STRIDE(i, n) d[idx[i]] = 0.0; }

// deterministic two-pass reductions (fixed grid, fixed tree): mode 0 dot, 1 sum|x|, 2 max|x|, 3 weighted dot
// sum_i w_i x_i y_i (shared-dof layouts count every dof once: w = 1 / number of ranks holding it)
template <int MODE>
__global__ void k_reduce_partial(const double *x, const double *y, size_t n, double *partial, const double *w = nullptr) {
  __shared__ double sh[256];
  double s = 0;
  GRID_STRIDE(i, n) {
    if (MODE == 0) s += x[i] * y[i];
    else if (MODE == 3) s += (w[i] * x[i]) * y[i];
    else if (MODE == 1) s += fabs(x[i]);
    else s = fmax(s, fabs(x[i]));
  }
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) sh[threadIdx.x] = MODE == 2 ? fmax(sh[threadIdx.x], sh[threadIdx.x + w]) : sh[threadIdx.x] + sh[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) partial[blockIdx.x] = sh[0];
}
template <int MODE>
__global__ void k_reduce_final(const double *partial, int np, double *out) {
  __shared__ double sh[256];
  double s = 0;
  for (int i = threadIdx.x; i < np; i += 256) s = MODE == 2 ? fmax(s, partial[i]) : s + partial[i];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) sh[threadIdx.x] = MODE == 2 ? fmax(sh[threadIdx.x], sh[threadIdx.x + w]) : sh[threadIdx.x] + sh[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = sh[0];
}

static double *g_partials[64] = {};  // per device: 1024 partials + 1 result
static const int kReduceBlocks = 592;  // 148 SMs x 4

static int partial_buffer(double **p) {
  int dev = 0;
  B200_CHECK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return set_error_msg("device ordinal out of range");
  if (!g_partials[dev]) B200_CHECK(cudaMalloc(&g_partials[dev], sizeof(double) * 1032));
  *p = g_partials[dev];
  return 0;
}

template <int MODE>
static int reduce(const double *x, const double *y, size_t n, double *dresult, const double *w = nullptr) {
  double *g_partial;
  if (int rc = partial_buffer(&g_partial)) return rc;
  k_reduce_partial<MODE><<<kReduceBlocks, 256, 0, g_stream>>>(x, y, n, g_partial, w);
  B200_LAUNCH_CHECK("k_reduce_partial");
  k_reduce_final<MODE><<<1, 256, 0, g_stream>>>(g_partial, kReduceBlocks, dresult);
  B200_LAUNCH_CHECK("k_reduce_final");
  return 0;
}
template <int MODE>
static int reduce_host(const double *x, const double *y, size_t n, double *hresult) {
  double *g_partial;
  if (int rc = partial_buffer(&g_partial)) return rc;
  if (int rc = reduce<MODE>(x, y, n, g_partial + 1024)) return rc;
  B200_CHECK(cudaMemcpyAsync(hresult, g_partial + 1024, sizeof(double), cudaMemcpyDeviceToHost, g_stream));
  B200_CHECK(cudaStreamSynchronize(g_stream));
  return 0;
}
}  // namespace b200

using namespace b200;

extern "C" {

int b200_device_count(int *count) { B200_CHECK(cudaGetDeviceCount(count)); return 0; }
int b200_set_device(int dev) { B200_CHECK(cudaSetDevice(dev)); return 0; }
int b200_get_device(int *dev) { B200_CHECK(cudaGetDevice(dev)); return 0; }
int b200_set_stream(void *s) { g_stream = (cudaStream_t)s; return 0; }
void *b200_get_stream(void) { return (void *)g_stream; }
int b200_sync(void) { B200_CHECK(cudaStreamSynchronize(g_stream)); return 0; }
const char *b200_last_error(void) { return g_err; }
int b200_device_name(char *buf, int len) {
  int dev; cudaDeviceProp p;
  B200_CHECK(cudaGetDevice(&dev));
  B200_CHECK(cudaGetDeviceProperties(&p, dev));
  snprintf(buf, len, "%s (sm_%d%d, %d SMs)", p.name, p.major, p.minor, p.multiProcessorCount);
  return 0;
}
int b200_sm_count(int *count) {
  int dev;
  B200_CHECK(cudaGetDevice(&dev));
  B200_CHECK(cudaDeviceGetAttribute(count, cudaDevAttrMultiProcessorCount, dev));
  return 0;
}

int b200_malloc(void **dptr, size_t bytes) { B200_CHECK(cudaMalloc(dptr, bytes ? bytes : 8)); return 0; }
int b200_free(void *dptr) { if (dptr) B200_CHECK(cudaFree(dptr)); return 0; }
int b200_malloc_host(void **hptr, size_t bytes) { B200_CHECK(cudaMallocHost(hptr, bytes ? bytes : 8)); return 0; }
int b200_free_host(void *hptr) { if (hptr) B200_CHECK(cudaFreeHost(hptr)); return 0; }
int b200_memset(void *dptr, int value, size_t bytes) { B200_CHECK(cudaMemsetAsync(dptr, value, bytes, g_stream)); return 0; }
int b200_memcpy_h2d(void *d, const void *h, size_t bytes) {
  B200_CHECK(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, g_stream));
  return 0;
}
int b200_memcpy_d2h(void *h, const void *d, size_t bytes) {
  B200_CHECK(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, g_stream));
  B200_CHECK(cudaStreamSynchronize(g_stream));
  return 0;
}
int b200_memcpy_d2d(void *d, const void *s, size_t bytes) {
  B200_CHECK(cudaMemcpyAsync(d, s, bytes, cudaMemcpyDeviceToDevice, g_stream));
  return 0;
}
int b200_pointer_is_device(const void *p, int *is_device) {
  cudaPointerAttributes at;
  cudaError_t e = cudaPointerGetAttributes(&at, p);
  if (e != cudaSuccess) { cudaGetLastError(); *is_device = 0; return 0; }
  *is_device = at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
  return 0;
}

unsigned long long b200_launch_count(void) { return g_launches; }
void b200_launch_count_reset(void) { g_launches = 0; }

#define VEC_KERNEL(call, n)                          \
  do {                                               \
    if ((n) == 0) return 0;                          \
    call;                                            \
    B200_LAUNCH_CHECK(#call);                        \
    return 0;                                        \
  } while (0)

int b200_vec_set(double *d, double v, size_t n) {
  if (v == 0.0) { if (n) B200_CHECK(cudaMemsetAsync(d, 0, n * sizeof(double), g_stream)); return 0; }
  VEC_KERNEL((k_set<<<grid_for(n, 256), 256, 0, g_stream>>>(d, v, n)), n);
}
int b200_vec_reciprocal(double *d, size_t n) { VEC_KERNEL((k_recip<<<grid_for(n, 256), 256, 0, g_stream>>>(d, n)), n); }
int b200_vec_scale(double *d, double a, size_t n) { VEC_KERNEL((k_scale<<<grid_for(n, 256), 256, 0, g_stream>>>(d, a, n)), n); }
int b200_vec_axpy(double *y, double a, const double *x, size_t n) { VEC_KERNEL((k_axpy<<<grid_for(n, 256), 256, 0, g_stream>>>(y, a, x, n)), n); }
int b200_vec_aypx(double *y, double a, const double *x, size_t n) { VEC_KERNEL((k_aypx<<<grid_for(n, 256), 256, 0, g_stream>>>(y, a, x, n)), n); }
int b200_vec_axpby(double *z, double a, const double *x, double b, const double *y, size_t n) {
  VEC_KERNEL((k_axpby<<<grid_for(n, 256), 256, 0, g_stream>>>(z, a, x, b, y, n)), n);
}
int b200_vec_pointwise_mult(double *w, const double *x, const double *y, size_t n) {
  VEC_KERNEL((k_pmult<<<grid_for(n, 256), 256, 0, g_stream>>>(w, x, y, n)), n);
}
int b200_vec_dot(const double *x, const double *y, size_t n, double *dresult) { return reduce<0>(x, y, n, dresult); }
int b200_vec_dot_weighted(const double *w, const double *x, const double *y, size_t n, double *dresult) {
  return reduce<3>(x, y, n, dresult, w);
}
int b200_vec_dot_host(const double *x, const double *y, size_t n, double *hresult) { return reduce_host<0>(x, y, n, hresult); }
int b200_vec_norm_host(const double *x, size_t n, int norm_type, double *hresult) {
  int rc;
  if (norm_type == 0) return reduce_host<1>(x, x, n, hresult);
  if (norm_type == 2) return reduce_host<2>(x, x, n, hresult);
  rc = reduce_host<0>(x, x, n, hresult);
  if (!rc) *hresult = sqrt(*hresult);
  return rc;
}
int b200_gather(double *dst, const double *src, const int *idx, size_t n) { VEC_KERNEL((k_gather<<<grid_for(n, 256), 256, 0, g_stream>>>(dst, src, idx, n)), n); }
int b200_scatter_set(double *dst, const int *idx, const double *src, size_t n) { VEC_KERNEL((k_scatter_set<<<grid_for(n, 256), 256, 0, g_stream>>>(dst, idx, src, n)), n); }
int b200_scatter_add(double *dst, const int *idx, const double *src, size_t n) { VEC_KERNEL((k_scatter_add<<<grid_for(n, 256), 256, 0, g_stream>>>(dst, idx, src, n)), n); }
int b200_gather_or_zero(double *dst, const double *src, const int *idx, size_t n) { VEC_KERNEL((k_gather_or_zero<<<grid_for(n, 256), 256, 0, g_stream>>>(dst, src, idx, n)), n); }
int b200_copy_where(double *dst, const double *src, const int *idx, size_t n) { VEC_KERNEL((k_copy_where<<<grid_for(n, 256), 256, 0, g_stream>>>(dst, src, idx, n)), n); }
int b200_vec_axpy_dev(double *y, const double *x, size_t n, const double *num, const double *den, double sign) {
  VEC_KERNEL((k_axpy_dev<<<grid_for(n, 256), 256, 0, g_stream>>>(y, x, n, num, den, sign)), n);
}
int b200_vec_aypx_dev(double *y, const double *x, size_t n, const double *num, const double *den) {
  VEC_KERNEL((k_aypx_dev<<<grid_for(n, 256), 256, 0, g_stream>>>(y, x, n, num, den)), n);
}
int b200_pcg_update(double *x, double *r, double *z, const double *p, const double *Ap, const double *dinv, size_t n,
                    const double *rz, const double *pAp) {
  VEC_KERNEL((k_pcg_update<<<grid_for(n, 256), 256, 0, g_stream>>>(x, r, z, p, Ap, dinv, n, rz, pAp)), n);
}
int b200_cheb_init(double *x, const double *r, double *d, const double *dinv, double inv_theta, int zero_guess, size_t n) {
  VEC_KERNEL((k_cheb_init<<<grid_for(n, 256), 256, 0, g_stream>>>(x, r, d, dinv, inv_theta, zero_guess, n)), n);
}
int b200_cheb_step(double *x, double *r, double *d, const double *Ad, const double *dinv, double c1, double c2, size_t n) {
  VEC_KERNEL((k_cheb_step<<<grid_for(n, 256), 256, 0, g_stream>>>(x, r, d, Ad, dinv, c1, c2, n)), n);
}
int b200_lattice_prolong(int Ncx, int Ncy, int Ncz, const double *xc, double *xf) {
  const size_t n = (size_t)3 * (2 * Ncx - 1) * (2 * Ncy - 1) * (2 * Ncz - 1);
  VEC_KERNEL((k_lattice_prolong<<<grid_for(n, 256), 256, 0, g_stream>>>(Ncx, Ncy, Ncz, xc, xf)), n);
}
int b200_lattice_restrict(int Ncx, int Ncy, int Ncz, const double *xf, double *xc) {
  const size_t n = (size_t)3 * Ncx * Ncy * Ncz;
  VEC_KERNEL((k_lattice_restrict<<<grid_for(n, 256), 256, 0, g_stream>>>(Ncx, Ncy, Ncz, xf, xc)), n);
}
int b200_stencil27_spmv(int Nx, int Ny, int Nz, const double *vals, const double *x, double *y) {
  const size_t n = (size_t)3 * Nx * Ny * Nz;
  VEC_KERNEL((k_stencil27_spmv<<<grid_for(n, 128), 128, 0, g_stream>>>(Nx, Ny, Nz, vals, x, y)), n);
}
int b200_ell_spmv(size_t n, int nslots, const int *cols, const double *vals, const double *x, double *y) {
  VEC_KERNEL((k_ell_spmv<<<grid_for(n, 128), 128, 0, g_stream>>>(n, nslots, cols, vals, x, y)), n);
}
int b200_fill_strided(double *d, double v, size_t n, size_t stride, size_t count) {
  VEC_KERNEL((k_fill_strided<<<grid_for(n * count, 256), 256, 0, g_stream>>>(d, v, n, stride, count)), n * count);
}
int b200_mask_zero(double *d, const int *idx, size_t n) { VEC_KERNEL((k_mask_zero<<<grid_for(n, 256), 256, 0, g_stream>>>(d, idx, n)), n); }

// ---------------------------------------------------------------------------------------------------
// Host-resident L-vectors (-memtype host, matops.c:40-50): CeedOperatorApply as a three-stage pipeline
//   copy engine 1: x chunks host -> device | SMs: fused kernel on element chunks | copy engine 2: finished y rows -> host
// The element range is cut into chunks; chunk c needs the input prefix [0, in_need[c]) and, once its kernel has
// run, the output prefix [0, out_final[c]) can receive no more contributions (both tables are derived from the
// offsets by the caller, so ANY numbering is handled correctly; only ordered ones overlap).  PCIe is full duplex,
// so the apply costs ~max(H2D, D2H) instead of H2D + kernel + D2H.  Both host arrays must be page-locked.
int b200_host_is_pinned(const void *p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return at.type == cudaMemoryTypeHost;
}

int b200_apply_hostpipe(int jacobian, int problem, const b200_physics *phys, int nelem, int P, int Q,
                        const double *hB, const double *hD, const int *d_offsets, const double *d_qa,
                        double *d_gradu, const double *h_x, double *d_x, double *h_y, double *d_y, size_t lsize,
                        int nchunks, const int *chunk_end, const size_t *in_need, const size_t *out_final) {
  enum { MAXC = 64 };
  static cudaStream_t s_in = nullptr, s_out = nullptr;
  static cudaEvent_t ev_in[MAXC], ev_k[MAXC], ev_start;
  static int pipe_device = -1;
  if (nchunks < 1 || nchunks > MAXC) return b200::set_error_msg("b200_apply_hostpipe: chunk count out of range");
  int dev = 0;
  B200_CHECK(cudaGetDevice(&dev));
  if (s_in && dev != pipe_device)
    return b200::set_error_msg("b200_apply_hostpipe: the process changed its CUDA device after the first host-vector apply "
                               "(one process per GPU is the supported model)");
  if (!s_in) {
    pipe_device = dev;
    B200_CHECK(cudaStreamCreateWithFlags(&s_in, cudaStreamNonBlocking));
    B200_CHECK(cudaStreamCreateWithFlags(&s_out, cudaStreamNonBlocking));
    for (int i = 0; i < MAXC; i++) {
      B200_CHECK(cudaEventCreateWithFlags(&ev_in[i], cudaEventDisableTiming));
      B200_CHECK(cudaEventCreateWithFlags(&ev_k[i], cudaEventDisableTiming));
    }
    B200_CHECK(cudaEventCreateWithFlags(&ev_start, cudaEventDisableTiming));
  }
  const int P3 = P * P * P, Q3 = Q * Q * Q;
  const int nc = jacobian ? b200_jcache_ncomp(problem) : 10;
  if (nc < 0) return b200::set_error_msg("b200_apply_hostpipe: unknown problem");
  // everything already queued on the compute stream (zeroing of y, earlier users of x) comes first
  B200_CHECK(cudaEventRecord(ev_start, g_stream));
  B200_CHECK(cudaStreamWaitEvent(s_in, ev_start, 0));
  B200_CHECK(cudaStreamWaitEvent(s_out, ev_start, 0));
  size_t copied = 0, sent = 0;
  int e0 = 0;
  for (int c = 0; c < nchunks; c++) {
    const bool last = c == nchunks - 1;
    size_t need = last ? lsize : in_need[c];
    if (need > lsize) need = lsize;
    if (need > copied) {
      B200_CHECK(cudaMemcpyAsync(d_x + copied, h_x + copied, (need - copied) * sizeof(double), cudaMemcpyHostToDevice, s_in));
      copied = need;
    }
    B200_CHECK(cudaEventRecord(ev_in[c], s_in));
    B200_CHECK(cudaStreamWaitEvent(g_stream, ev_in[c], 0));
    const int ne = chunk_end[c] - e0;
    if (ne > 0) {
      const int rc = jacobian
          ? b200_apply_jacobian(problem, phys, ne, P, Q, hB, hD, d_offsets + (size_t)e0 * P3, d_qa + (size_t)e0 * nc * Q3, d_x, d_y, nullptr)
          : b200_apply_residual(problem, phys, ne, P, Q, hB, hD, d_offsets + (size_t)e0 * P3, d_qa + (size_t)e0 * nc * Q3,
                                d_gradu ? d_gradu + (size_t)e0 * 9 * Q3 : nullptr, d_x, d_y, nullptr);
      if (rc) return rc;
    }
    B200_CHECK(cudaEventRecord(ev_k[c], g_stream));
    B200_CHECK(cudaStreamWaitEvent(s_out, ev_k[c], 0));
    size_t fin = last ? lsize : out_final[c];
    if (fin > lsize) fin = lsize;
    if (fin > sent) {
      B200_CHECK(cudaMemcpyAsync(h_y + sent, d_y + sent, (fin - sent) * sizeof(double), cudaMemcpyDeviceToHost, s_out));
      sent = fin;
    }
    e0 = chunk_end[c];
  }
  B200_CHECK(cudaStreamSynchronize(s_out));  // the libCEED call is synchronous for host-visible results
  B200_CHECK(cudaStreamSynchronize(g_stream));
  return 0;
}

// FP64 pipe probe (SURVEY 8(d): "measure with a DFMA microbenchmark"): 8 independent DFMA chains per thread.
int b200_fp64_probe(double *dfma_per_second) {
  const int iters = 4096, nblk = 148 * 16, nthr = 256;
  double *sink = nullptr;
  B200_CHECK(cudaMalloc(&sink, sizeof(double) * nblk * nthr));
  cudaEvent_t e0, e1;
  B200_CHECK(cudaEventCreate(&e0));
  B200_CHECK(cudaEventCreate(&e1));
  k_fp64_probe<<<nblk, nthr, 0, g_stream>>>(sink, iters, 1.0000001);   // warm-up
  B200_CHECK(cudaEventRecord(e0, g_stream));
  for (int r = 0; r < 4; r++) k_fp64_probe<<<nblk, nthr, 0, g_stream>>>(sink, iters, 1.0000001);
  B200_CHECK(cudaEventRecord(e1, g_stream));
  B200_CHECK(cudaEventSynchronize(e1));
  B200_LAUNCH_CHECK("k_fp64_probe");
  float ms = 0;
  B200_CHECK(cudaEventElapsedTime(&ms, e0, e1));
  *dfma_per_second = 4.0 * 8.0 * iters * (double)nblk * nthr / (ms * 1e-3);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  B200_CHECK(cudaFree(sink));
  return 0;
}

int b200_elems_per_block(int Q) { return elems_per_block(Q); }
int b200_strided_layout_q(int elemsize) {
  for (int Q = 2; Q <= 8; Q++)
    if (Q * Q * Q == elemsize) return Q;
  return 0;
}

}  // extern "C"
