// Shared helpers for the /gpu/b200 CUDA layer (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "b200_kernels.h"

namespace b200 {

extern cudaStream_t g_stream;
extern unsigned long long g_launches;
int set_error(cudaError_t e, const char *what);
int set_error_msg(const char *msg);
// Gc = D pinv(B), Gc B = D: the collocated derivative of a tensor basis (b200_fused.cu); != 0 if B is rank-deficient
int collocated_grad_1d(int P, int Q, const double *B, const double *D, double *Gc);

#define B200_CHECK(call)                                   \
  do {                                                     \
    cudaError_t _e = (call);                               \
    if (_e != cudaSuccess) return b200::set_error(_e, #call); \
  } while (0)

#define B200_LAUNCH_CHECK(name)                            \
  do {                                                     \
    b200::g_launches++;                                    \
    cudaError_t _e = cudaGetLastError();                   \
    if (_e != cudaSuccess) return b200::set_error(_e, name); \
  } while (0)

// elements per thread block of the fused kernels == group size of the q-blocked layout
// (Q >= 4: 4 elements x Q^2 threads = 64 / 100 threads per CTA: many small independent CTAs per SM
// hide the per-stage barriers and load latencies better than fewer large ones -- measured)
#ifndef B200_EB_BIG
#define B200_EB_BIG 4
#endif
__host__ __device__ constexpr int elems_per_block(int Q) { return Q <= 3 ? 16 : B200_EB_BIG; }

// Index of (element e, component c, point q) in a q-blocked backend-strided vector:
// groups of EB elements; inside a group holding ebn elements (ebn = EB except in the tail)
//   [comp][qx][t = qy + Q*qz][element-in-group]
// so that the fused kernels' lane id (tid = t*ebn + e) walks contiguous memory.
__host__ __device__ inline size_t qblocked_index(int nelem, int ncomp, int Q, int e, int c, int q) {
  const int EB = elems_per_block(Q), T = Q * Q, Q3 = Q * Q * Q;
  const int g = e / EB, ei = e - g * EB;
  const int rem = nelem - g * EB;
  const int ebn = rem < EB ? rem : EB;
  return (size_t)g * EB * ncomp * Q3 + (size_t)(c * Q + q % Q) * (ebn * T) + (size_t)(q / Q) * ebn + ei;
}

// ---------------------------------------------------------------------------------
// material constants derived once on the host from Physics {nu, E}
// (qfunctions/hyperFS.h:164-167, qfunctions/linElas.h:127-133)
// ---------------------------------------------------------------------------------
struct Material {
  double nu, E;
  double TwoMu, mu, lambda;
  double le_c1, le_c2, le_c3;  // linElas: ss(1-nu), ss*nu, ss(1-2nu)/4
};

inline Material make_material(const b200_physics *p) {
  Material m;
  m.nu = p->nu;
  m.E = p->E;
  m.TwoMu = m.E / (1 + m.nu);
  m.mu = m.TwoMu / 2;
  const double Kbulk = m.E / (3 * (1 - 2 * m.nu));
  m.lambda = (3 * Kbulk - m.TwoMu) / 3;
  const double ss = m.E / ((1 + m.nu) * (1 - 2 * m.nu));
  m.le_c1 = ss * (1 - m.nu);
  m.le_c2 = ss * m.nu;
  m.le_c3 = ss * (1 - 2 * m.nu) * 0.5 * 0.5;
  return m;
}

}  // namespace b200
