// Fused matrix-free operator kernels of the /gpu/b200 backend (sm_100a, FP64).
//
//   y_L += E^T G^T D(q-data) G E x_L          one launch per CeedOperatorApply
//
// replaces, for the residual / Jacobian operators the reference builds in
// /root/reference/src/setuplibceed.c:518-542 and :818-839, the whole backend side of
// CeedOperatorApply called from ApplyLocalCeedOp (/root/reference/src/matops.c:46):
// offsets gather, tensor-product gradient, QFunction, transposed gradient, scatter-add.
//
// Mapping.  Q*Q threads per element, EB elements per CTA (EB*Q*Q ~ 128 threads).  A thread
// always owns one LINE of the Q^3 (or P^3) lattice in registers and contracts it against the
// basis matrix, which is a kernel parameter (constant bank, immediate operand of DFMA): one
// LDS/STS per five DFMAs instead of one per DFMA.  Between stages the lattice is re-oriented
// through shared memory:
//
//   gather (z-lines)  --B_z-->  y-lines --B_y-->  x-lines --B_x--> u~ at quadrature points
//   x-lines: d/dx in registers;  y-lines, z-lines: d/dy, d/dz with the collocated
//   derivative matrix Gc (Gc B = D);  x-lines again: QFunction at the thread's Q points,
//   streaming the q-blocked per-point data straight from HBM (fully coalesced);
//   then the exact transpose back, the nodal output written interlaced [node][component],
//   and a scatter sweep in L-vector order (FP64 atomics, or plain stores to an E-vector
//   in deterministic mode).
//
// FP64 work at P=Q=5: 12 line stages x 1875 DFMA + 125 x ~150 (hyperFS Jacobian from the
// Jacobian cache) ~ 41 k per element, vs ~100 k for libCEED-style 9-contraction gradients
// around the unmodified QFunction.  The binding unit is the L1TEX data pipe (25 lattice passes
// through shared memory + the stream + gather/scatter: 86 % busy); see DESIGN.md section 3 and
// profiles/r2_k_fused_apply_full.md.
#include "b200_qf.cuh"

#include <stdlib.h>
#include <string.h>

namespace b200 {

template <int P, int Q> struct Mats {
  double B[Q * P];   // interp1d  [Q][P]
  double Gc[Q * Q];  // collocated derivative at the quadrature points, Gc * B = grad1d
};

template <int Q> struct Cfg {
  static constexpr int T = Q * Q;
  static constexpr int EB = elems_per_block(Q);
  static constexpr int NT = ((T * EB + 31) / 32) * 32;
  static constexpr int Q3 = Q * Q * Q;
  // Shared-memory lattice with ODD strides (1, QP, QP^2) and lanes ordered element-fastest
  // (tid = t*EB + e): a half-warp then holds EB=16 elements of one line, or 16/EB neighbouring
  // lines of EB elements whose lattice offsets are distinct mod 16/EB; with the element stride SE
  // odd (EB=16) or = 16/EB mod 16 (EB=8, 4) every 64-bit shared access of every line orientation
  // is bank-conflict free (checked exhaustively in tests/test_abi_and_layout.py).
  static constexpr int QP = (Q % 2) ? Q : Q + 1;
  static constexpr int SY = QP, SZ = QP * QP, SC = QP * QP * QP;
  static constexpr int SE0 = 9 * SC;
  static constexpr int SEM = 16 / EB;  // EB=8: SE = 2 mod 16, EB=4: SE = 4 mod 16, EB=16: odd
  static constexpr int SE = EB == 16 ? (SE0 | 1) : SE0 + ((SEM - SE0 % 16) + 16) % 16;
  static constexpr size_t SMEM = (size_t)EB * SE * sizeof(double);
};

#define IDX(c, x, y, z) ((c) * SC + (z) * SZ + (y) * SY + (x))

// Shared-memory extents of the fused apply kernels: three gradient lattices of three components each.
// (A padded component stride that made the final scatter sweep conflict-free was measured SLOWER, 1.26 vs 1.13 ms at
// P = Q = 5: 42 kB per CTA pushes five resident CTAs past the 196 kB shared-memory carve-out and leaves the gather
// 28 kB of L1 instead of 60 kB.  The sweep is made conflict-free without extra memory instead: the last stage writes
// its nodal output interlaced, [node][component], into the lattices that are free by then.)
__host__ __device__ constexpr int odd_extent(int Q) { return (Q % 2) ? Q : Q + 1; }
__host__ __device__ constexpr int apply_sc(int P, int Q) { return odd_extent(Q) * odd_extent(Q) * odd_extent(Q); }
__host__ __device__ constexpr int apply_se(int Q, int SC) {
  return elems_per_block(Q) == 16 ? ((9 * SC) | 1) : 9 * SC + ((16 / elems_per_block(Q) - (9 * SC) % 16) + 16) % 16;
}

// one thread asks the L2 to fetch this CTA's whole slab of per-point data (contiguous in the
// q-blocked layout) while the CTA is busy with the gather and the interpolation stages
__device__ __forceinline__ void l2_prefetch_bulk(const void *p, unsigned bytes) {
  bytes &= ~15u;
  if (bytes) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}

// per-point stream: read once, never reused.  Default: ld.global.cs (evict-first in L1 and L2).
// B200_STREAM_NOALLOC (tuning build): do not allocate the line in L1 at all -- keeps the small L1
// (60 kB beside 196 kB of shared memory) for the gather of x and the offsets.
__device__ __forceinline__ double ld_stream(const double *p) {
#ifdef B200_STREAM_NOALLOC
  double v;
  asm volatile("ld.global.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
#else
  return __ldcs(p);
#endif
}

enum { MODE_RESIDUAL = 0, MODE_JACOBIAN = 1 };

// FULL: every CTA of the launch owns a complete group of EB elements, so the plane stride of the q-blocked
// per-point data is a compile-time constant and every stream load is [base + immediate] (the tail group of a
// launch, if any, runs through the FULL = false instantiation in a second one-CTA launch).
template <int P, int Q, int PROB, int MODE, bool FULL>
// min CTAs/SM: 5 x 128 threads caps the Jacobian kernels at 96 registers (no spills at P=Q=5) and
// measured 3.5 % faster than 4 x 128 regs; the residual kernels keep all registers
// (residual kernels: 4 CTAs/SM (128 registers, a few spilled words) measured 20 % faster than 1-2 CTAs at 228 registers)
#ifndef B200_JAC_CTAS
#define B200_JAC_CTAS 5
#endif
#ifndef B200_RES_CTAS
#define B200_RES_CTAS 4
#endif
#ifndef B200_RES_AHEAD
#define B200_RES_AHEAD 1
#endif
#ifndef B200_RES_ROLLED
#define B200_RES_ROLLED 0
#endif
#ifndef B200_JAC_ROLLED
#define B200_JAC_ROLLED 0
#endif
__global__ void __launch_bounds__(Cfg<Q>::NT, MODE == MODE_JACOBIAN ? (Cfg<Q>::NT <= 128 ? B200_JAC_CTAS : 2) : (Cfg<Q>::NT <= 128 ? B200_RES_CTAS : 1))
k_fused_apply(const __grid_constant__ Mats<P, Q> m, const __grid_constant__ Material mt, int nelem,
              const int *__restrict__ offsets, const double *__restrict__ qa,
              double *__restrict__ gradu, const double *__restrict__ x, double *__restrict__ y,
              const unsigned *__restrict__ scat_tab, int offsets_ahead, double *__restrict__ evec, int x_ahead, int slab_ahead) {
  constexpr int T = Cfg<Q>::T, EB = Cfg<Q>::EB, Q3 = Cfg<Q>::Q3, P3 = P * P * P;
  constexpr int SY = Cfg<Q>::SY, SZ = Cfg<Q>::SZ, SC = apply_sc(P, Q), SE = apply_se(Q, SC);
  constexpr int NC = MODE == MODE_JACOBIAN ? JCache<PROB>::N : 10;
  extern __shared__ double smem[];
  const int tid = threadIdx.x;
  const int t = tid / EB, eb = tid - t * EB, a = t % Q, b = t / Q;
  const int blk = blockIdx.x;
  const int rem = nelem - blk * EB;
  const int ebn = FULL ? EB : (rem < EB ? rem : EB);
  const bool act = t < T && (FULL || eb < ebn);
  const int e = blk * EB + eb;
  double *R0 = smem + eb * SE, *R1 = R0 + 3 * SC, *R2 = R1 + 3 * SC;
  // per-point data of this CTA: slab base + lane offset, plane stride (q-blocked layout)
  const size_t ebt = FULL ? (size_t)(EB * T) : (size_t)ebn * T;
  const double *qlane = qa + (size_t)blk * EB * NC * Q3 + (FULL ? tid : t * ebn + eb);
  // slab_ahead = 0: the CTA asks for its OWN slab at its start (it needs it ~4 us later, in the point-function stage);
  // > 0 (full groups only): for the slab of the CTA that many groups later, so that a slab is in L2 before its CTA starts
  if (tid == 0) {
    if (!FULL || slab_ahead <= 0 || blk < slab_ahead)
      l2_prefetch_bulk(qa + (size_t)blk * EB * NC * Q3, (unsigned)(ebt * Q * NC * sizeof(double)));
    if (FULL && slab_ahead > 0 && (long long)(blk + slab_ahead + 1) * EB <= nelem)
      l2_prefetch_bulk(qa + (size_t)(blk + slab_ahead) * EB * NC * Q3, (unsigned)(ebt * Q * NC * sizeof(double)));
  }
  // ... and the element offsets of a CTA that starts about one wave of resident CTAs later: its gather then
  // begins with an L2 hit instead of a DRAM round trip in front of the dependent loads of x
  if (FULL && tid == 32 && offsets_ahead > 0 && (long long)(blk + offsets_ahead + 1) * EB <= nelem)
    l2_prefetch_bulk(offsets + (size_t)(blk + offsets_ahead) * EB * P3, (unsigned)(EB * P3 * sizeof(int)));

  int *soff = reinterpret_cast<int *>(smem + EB * SE);
  // ---- phase 0: gather node z-lines, contract z with B
  if (act && a < P && b < P) {
    double r[3][P];
    const int *off = offsets + (size_t)e * P3 + b * P + a;
    int o[P];
#pragma unroll
    for (int k = 0; k < P; k++) o[k] = __ldg(off + k * P * P);
    // the L-vector entries a CTA x_ahead groups later will gather: its offsets are in L2 already (prefetched by an
    // earlier CTA), so this costs one L2 round trip that nothing waits for; the later CTA's dependent second load
    // then finds x in L2 instead of DRAM
    if (FULL && x_ahead > 0 && (long long)(blk + x_ahead + 1) * EB <= nelem) {
      const int *offn = off + (size_t)x_ahead * EB * P3;
      int on[P];
#pragma unroll
      for (int k = 0; k < P; k++) on[k] = __ldg(offn + k * P * P);
#pragma unroll
      for (int k = 0; k < P; k++) asm volatile("prefetch.global.L2 [%0];" ::"l"(x + on[k]));
    }
#pragma unroll
    for (int k = 0; k < P; k++) {
      soff[eb * P3 + (k * P + b) * P + a] = o[k];  // parked for the scatter at the end
#pragma unroll
      for (int c = 0; c < 3; c++) r[c][k] = __ldg(x + o[k] + c);
    }
#pragma unroll
    for (int c = 0; c < 3; c++)
#pragma unroll
      for (int qz = 0; qz < Q; qz++) {
        double s = 0;
#pragma unroll
        for (int k = 0; k < P; k++) s += m.B[qz * P + k] * r[c][k];
        R0[IDX(c, a, b, qz)] = s;
      }
  }
  __syncthreads();
  // ---- phase 1: y-lines (a = i, b = qz), contract y with B
  if (act && a < P) {
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double in[P];
#pragma unroll
      for (int j = 0; j < P; j++) in[j] = R0[IDX(c, a, j, b)];
#pragma unroll
      for (int qy = 0; qy < Q; qy++) {
        double s = 0;
#pragma unroll
        for (int j = 0; j < P; j++) s += m.B[qy * P + j] * in[j];
        R1[IDX(c, a, qy, b)] = s;
      }
    }
  }
  __syncthreads();
  // ---- phase 2: x-lines (a = qy, b = qz), contract x with B; d/dx in registers
  double Hx[3][Q];
  if (act) {
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double in[P], ut[Q];
#pragma unroll
      for (int i = 0; i < P; i++) in[i] = R1[IDX(c, i, a, b)];
#pragma unroll
      for (int qx = 0; qx < Q; qx++) {
        double s = 0;
#pragma unroll
        for (int i = 0; i < P; i++) s += m.B[qx * P + i] * in[i];
        ut[qx] = s;
        R0[IDX(c, qx, a, b)] = s;
      }
#pragma unroll
      for (int qx = 0; qx < Q; qx++) {
        double s = 0;
#pragma unroll
        for (int mm = 0; mm < Q; mm++) s += m.Gc[qx * Q + mm] * ut[mm];
        Hx[c][qx] = s;
      }
    }
  }
  __syncthreads();
  // ---- phase 3: y-lines (a = qx, b = qz): d/dy -> R1;  phase 4: z-lines (a = qx, b = qy): d/dz -> R2
  // per-point data of the NEXT quadrature point: loads stay in flight under the math.  (A/B at 64^3, hyperFS residual,
  // 4 CTAs/SM at 128 registers: look-ahead with 40 B of spills 1.44 ms, no look-ahead and no spills 1.52 ms, 3 CTAs/SM at
  // 158 registers with look-ahead 1.53 ms: B200_RES_AHEAD / B200_RES_CTAS.)
  constexpr bool AHEAD = B200_RES_AHEAD || !(MODE == MODE_RESIDUAL && PROB == B200_PROB_HYPERFS);
  double qn[NC];
  if (act) {
    if (AHEAD) {
#pragma unroll
      for (int n = 0; n < NC; n++) qn[n] = ld_stream(qlane + (size_t)(n * Q) * ebt);
    }
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double in[Q];
#pragma unroll
      for (int mm = 0; mm < Q; mm++) in[mm] = R0[IDX(c, a, mm, b)];
#pragma unroll
      for (int qy = 0; qy < Q; qy++) {
        double s = 0;
#pragma unroll
        for (int mm = 0; mm < Q; mm++) s += m.Gc[qy * Q + mm] * in[mm];
        R1[IDX(c, a, qy, b)] = s;
      }
#pragma unroll
      for (int mm = 0; mm < Q; mm++) in[mm] = R0[IDX(c, a, b, mm)];
#pragma unroll
      for (int qz = 0; qz < Q; qz++) {
        double s = 0;
#pragma unroll
        for (int mm = 0; mm < Q; mm++) s += m.Gc[qz * Q + mm] * in[mm];
        R2[IDX(c, a, b, qz)] = s;
      }
    }
  }
  __syncthreads();
  // ---- phase 5: QFunction at the Q points of this x-line; phase 6: d/dx^T in registers
  // ROLLED (tuning switch, OFF): the loop over the Q points of the line not unrolled.  Fully unrolled, the hyperFS
  // residual kernel is 3 120 instructions (50 kB), past the instruction-cache plateau, and ncu attributes 24 % of its
  // stall samples to instruction fetch (no_inst); rolled (the line values rotate through a register array with static
  // indices: Hx[.][0] is consumed, the array shifts left, the new W[.][0] enters at the end) it is 2 168 instructions --
  // but MEASURED SLOWER: residual 1.59 vs 1.45 ms, Jacobian 1.82 vs 1.13 ms at 64^3 (the scheduler loses the overlap of
  // one point's loads and stores with the next point's arithmetic).  Kept for the record.
  constexpr bool ROLLED = MODE == MODE_RESIDUAL ? (B200_RES_ROLLED != 0) : (B200_JAC_ROLLED != 0);
  if (act && ROLLED) {
    const double *qp = qlane;                                    // advances by one plane per point
    double *g1 = R1 + IDX(0, 0, a, b), *g2 = R2 + IDX(0, 0, a, b);
    double *gslab = (MODE == MODE_RESIDUAL && PROB != B200_PROB_LINELAS)
                        ? gradu + (size_t)blk * EB * 9 * Q3 + (FULL ? tid : t * ebn + eb) : nullptr;
#pragma unroll 1
    for (int qx = 0; qx < Q; qx++) {
      double qd[NC], H[3][3], W[3][3];
      if (AHEAD) {
#pragma unroll
        for (int n = 0; n < NC; n++) qd[n] = qn[n];
        if (qx + 1 < Q) {
#pragma unroll
          for (int n = 0; n < NC; n++) qn[n] = ld_stream(qp + (size_t)(n * Q + 1) * ebt);
        }
      } else {
#pragma unroll
        for (int n = 0; n < NC; n++) qd[n] = ld_stream(qp + (size_t)(n * Q) * ebt);
      }
#pragma unroll
      for (int c = 0; c < 3; c++) {
        H[c][0] = Hx[c][0];
        H[c][1] = g1[c * SC];
        H[c][2] = g2[c * SC];
      }
      if (MODE == MODE_JACOBIAN) {
        jacobian_point<PROB>(mt, qd, H, W);
      } else {
        double A[3][3], g[3][3];
#pragma unroll
        for (int mm = 0; mm < 3; mm++)
#pragma unroll
          for (int k = 0; k < 3; k++) A[mm][k] = qd[1 + 3 * mm + k];
        if (PROB == B200_PROB_LINELAS) {
          linelas_point(mt, qd[0], A, H, W);
        } else {
          if (PROB == B200_PROB_HYPERSS) hyperss_f_point(mt, qd[0], A, H, g, W);
          else hyperfs_f_point(mt, qd[0], A, H, g, W);
#pragma unroll
          for (int c = 0; c < 3; c++)
#pragma unroll
            for (int k = 0; k < 3; k++) __stcs(gslab + (size_t)((c * 3 + k) * Q) * ebt, g[c][k]);
          gslab += ebt;
        }
      }
#pragma unroll
      for (int c = 0; c < 3; c++) {
#pragma unroll
        for (int i = 0; i + 1 < Q; i++) Hx[c][i] = Hx[c][i + 1];
        Hx[c][Q - 1] = W[c][0];
        g1[c * SC] = W[c][1];
        g2[c * SC] = W[c][2];
      }
      qp += ebt;
      g1++;
      g2++;
    }
#pragma unroll
    for (int c = 0; c < 3; c++)
#pragma unroll
      for (int qx = 0; qx < Q; qx++) {
        double s = 0;
#pragma unroll
        for (int mm = 0; mm < Q; mm++) s += m.Gc[mm * Q + qx] * Hx[c][mm];
        R0[IDX(c, qx, a, b)] = s;
      }
  }
  if (act && !ROLLED) {
    double Wx[3][Q];
#pragma unroll
    for (int qx = 0; qx < Q; qx++) {
      double qd[NC], H[3][3], W[3][3];
      if (AHEAD) {
#pragma unroll
        for (int n = 0; n < NC; n++) qd[n] = qn[n];
        if (qx + 1 < Q) {
#pragma unroll
          for (int n = 0; n < NC; n++) qn[n] = ld_stream(qlane + (size_t)(n * Q + qx + 1) * ebt);
        }
      } else {
#pragma unroll
        for (int n = 0; n < NC; n++) qd[n] = ld_stream(qlane + (size_t)(n * Q + qx) * ebt);
      }
#pragma unroll
      for (int c = 0; c < 3; c++) {
        H[c][0] = Hx[c][qx];
        H[c][1] = R1[IDX(c, qx, a, b)];
        H[c][2] = R2[IDX(c, qx, a, b)];
      }
      if (MODE == MODE_JACOBIAN) {
        jacobian_point<PROB>(mt, qd, H, W);
      } else {
        double A[3][3], g[3][3];
#pragma unroll
        for (int mm = 0; mm < 3; mm++)
#pragma unroll
          for (int k = 0; k < 3; k++) A[mm][k] = qd[1 + 3 * mm + k];
        if (PROB == B200_PROB_LINELAS) {
          linelas_point(mt, qd[0], A, H, W);
        } else {
          if (PROB == B200_PROB_HYPERSS) hyperss_f_point(mt, qd[0], A, H, g, W);
          else hyperfs_f_point(mt, qd[0], A, H, g, W);
          double *gslab = gradu + (size_t)blk * EB * 9 * Q3 + (FULL ? tid : t * ebn + eb);
#pragma unroll
          for (int c = 0; c < 3; c++)
#pragma unroll
            for (int k = 0; k < 3; k++) __stcs(gslab + (size_t)((c * 3 + k) * Q + qx) * ebt, g[c][k]);
        }
      }
#pragma unroll
      for (int c = 0; c < 3; c++) {
        Wx[c][qx] = W[c][0];
        R1[IDX(c, qx, a, b)] = W[c][1];
        R2[IDX(c, qx, a, b)] = W[c][2];
      }
    }
#pragma unroll
    for (int c = 0; c < 3; c++)
#pragma unroll
      for (int qx = 0; qx < Q; qx++) {
        double s = 0;
#pragma unroll
        for (int mm = 0; mm < Q; mm++) s += m.Gc[mm * Q + qx] * Wx[c][mm];
        R0[IDX(c, qx, a, b)] = s;
      }
  }
  __syncthreads();
  // ---- phase 7: y-lines (a = qx, b = qz): R0 += Gc^T_y Wy
  if (act) {
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double in[Q];
#pragma unroll
      for (int mm = 0; mm < Q; mm++) in[mm] = R1[IDX(c, a, mm, b)];
#pragma unroll
      for (int qy = 0; qy < Q; qy++) {
        double s = R0[IDX(c, a, qy, b)];
#pragma unroll
        for (int mm = 0; mm < Q; mm++) s += m.Gc[mm * Q + qy] * in[mm];
        R0[IDX(c, a, qy, b)] = s;
      }
    }
  }
  __syncthreads();
  // ---- phase 8: z-lines (a = qx, b = qy): v~ = R0 + Gc^T_z Wz, then B^T along z -> R1
  if (act) {
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double in[Q], vt[Q];
#pragma unroll
      for (int mm = 0; mm < Q; mm++) in[mm] = R2[IDX(c, a, b, mm)];
#pragma unroll
      for (int qz = 0; qz < Q; qz++) {
        double s = R0[IDX(c, a, b, qz)];
#pragma unroll
        for (int mm = 0; mm < Q; mm++) s += m.Gc[mm * Q + qz] * in[mm];
        vt[qz] = s;
      }
#pragma unroll
      for (int k = 0; k < P; k++) {
        double s = 0;
#pragma unroll
        for (int qz = 0; qz < Q; qz++) s += m.B[qz * P + k] * vt[qz];
        R1[IDX(c, a, b, k)] = s;
      }
    }
  }
  __syncthreads();
  // ---- phase 9: y-lines (a = qx, b = k < P): B^T along y -> R2
  if (act && b < P) {
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double in[Q];
#pragma unroll
      for (int qy = 0; qy < Q; qy++) in[qy] = R1[IDX(c, a, qy, b)];
#pragma unroll
      for (int j = 0; j < P; j++) {
        double s = 0;
#pragma unroll
        for (int qy = 0; qy < Q; qy++) s += m.B[qy * P + j] * in[qy];
        R2[IDX(c, a, j, b)] = s;
      }
    }
  }
  __syncthreads();
  // ---- phase 10: x-lines (a = j < P, b = k < P): B^T along x -> nodal output, interlaced [node][component] at the
  // start of the element's region (lattices R0 and R1 are free: last read in phases 8 and 9): the scatter sweep
  // below then reads consecutive shared-memory words (no bank conflicts) in exactly L-vector order
  if (act && a < P && b < P) {
    double *Rn = R0 + ((b * P + a) * P) * 3;
    static_assert(3 * P3 <= 6 * SC, "interlaced nodal output must fit in the first two lattices");
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double in[Q];
#pragma unroll
      for (int qx = 0; qx < Q; qx++) in[qx] = R2[IDX(c, qx, a, b)];
#pragma unroll
      for (int i = 0; i < P; i++) {
        double s = 0;
#pragma unroll
        for (int qx = 0; qx < Q; qx++) s += m.B[qx * P + i] * in[qx];
        Rn[i * 3 + c] = s;
      }
    }
  }
  __syncthreads();
  // ---- scatter-add in L-vector order: flat sweep f = (element, node, component), component fastest, so
  // consecutive lanes hit consecutive L-vector entries (interlaced dofs) and one RED request touches few
  // sectors.  The (lattice index, offset index, component) of each f is the same for every CTA: it comes
  // from a small table (L1/L2 resident) instead of ~30 integer instructions of div/mod per entry.
  // All shared-memory reads of the sweep are issued before the first RED so that none waits behind one.
  {
    constexpr int NT = Cfg<Q>::NT, NIT = (EB * 3 * P3 + NT - 1) / NT;
    const int total = ebn * 3 * P3;
    unsigned u[NIT];
#pragma unroll
    for (int it = 0; it < NIT; it++) u[it] = (FULL && (it + 1) * NT <= EB * 3 * P3) || (tid + it * NT < total) ? __ldg(scat_tab + tid + it * NT) : 0u;
#ifdef B200_NO_BATCH_SCATTER
    if (!evec) {
#pragma unroll
      for (int it = 0; it < NIT; it++)
        if (tid + it * NT < total)
          atomicAdd(y + soff[(u[it] >> 16) & 0xFFFu] + (u[it] >> 28), smem[u[it] & 0xFFFFu]);
      return;
    }
#endif
    double val[NIT];
    int dst[NIT];
#pragma unroll
    for (int it = 0; it < NIT; it++) {
      val[it] = smem[u[it] & 0xFFFFu];
      dst[it] = soff[(u[it] >> 16) & 0xFFFu] + (int)(u[it] >> 28);
    }
    if (evec) {  // deterministic mode: element outputs [e][node][comp], summed in a fixed order by the caller
      double *ev = evec + (size_t)blk * EB * 3 * P3;
#pragma unroll
      for (int it = 0; it < NIT; it++)
        if ((FULL && (it + 1) * NT <= EB * 3 * P3) || tid + it * NT < total) ev[tid + it * NT] = val[it];
    } else {
#pragma unroll
      for (int it = 0; it < NIT; it++)
        if ((FULL && (it + 1) * NT <= EB * 3 * P3) || tid + it * NT < total) atomicAdd(y + dst[it], val[it]);
    }
  }
}

// -----------------------------------------------------------------------------------
// Jacobian cache build: point-wise over the q-blocked layout (same position in every
// component plane), coalesced.
// -----------------------------------------------------------------------------------
template <int PROB>
__global__ void k_jcache_build(int nelem, int Q, const double *__restrict__ qdata,
                               const double *__restrict__ gradu, double *__restrict__ jc) {
  constexpr int NJ = JCache<PROB>::N;
  const int EB = elems_per_block(Q), Q3 = Q * Q * Q, T = Q * Q;
  const size_t npts = (size_t)nelem * Q3;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < npts; i += (size_t)gridDim.x * blockDim.x) {
    // i enumerates positions group by group: i = g*EB*Q3 + r, r in [0, ebn*Q3)
    const size_t g = i / ((size_t)EB * Q3);
    const int r = (int)(i - g * EB * Q3);
    const long long rem = (long long)nelem - (long long)g * EB;
    const int ebn = rem < EB ? (int)rem : EB;
    const size_t plane = (size_t)ebn * T * Q;  // points per component plane in this group
    double qd[10], gu[9], out[NJ];
    const double *qp = qdata + g * EB * 10 * Q3 + r;
#pragma unroll
    for (int n = 0; n < 10; n++) qd[n] = __ldcs(qp + n * plane);
    if (PROB != B200_PROB_LINELAS) {
      const double *gp = gradu + g * EB * 9 * Q3 + r;
#pragma unroll
      for (int n = 0; n < 9; n++) gu[n] = __ldcs(gp + n * plane);
    }
    jcache_point<PROB>(qd, gu, out);
    double *jp = jc + g * EB * NJ * Q3 + r;
#pragma unroll
    for (int n = 0; n < NJ; n++) jp[n * plane] = out[n];
  }
}

// -----------------------------------------------------------------------------------
// Operator diagonal (CeedOperatorLinearAssembleDiagonal, matops.c:227; App. B.5):
//   diag_e[c][n] = sum_q sum_{d,d'} G_d[q,n] A_c[d'][d](q) G_d'[q,n]
// A_c = symmetric 3x3 point block in closed form (diag_blocks_point), G_d = Kronecker(B or D per axis), so
// each of the six distinct (d,d') terms is a 3-stage sum-factorised contraction with the element-wise
// products B.B, B.D, D.D.  Term t (Voigt order 00,11,22,12,02,01; off-diagonal terms count twice):
//   x-stage: S_t[i]    = sum_qx A_t(qx) Mx[sel_x(t)][qx][i]      (x-line owner, registers)
//   y-stage: Y_s[j]   += sum_qy S_t(qy) My[sel_y(t)][qy][j]      terms merged by their z selector s
//   z-stage: acc[k]   += sum_qz Y_s(qz) Mz[s][qz][k]
// The cache slab of the CTA is read once from HBM (component 0) and twice more through L2.
// -----------------------------------------------------------------------------------
template <int P, int Q> struct DiagMats {
  double M[3][Q * P];  // [0] B.B  [1] B.D  [2] D.D   (element-wise, [Q][P])
};

template <int P, int Q, int PROB, bool FULL>
#ifndef B200_DIAG_THREADS
#define B200_DIAG_THREADS 384
#endif
__global__ void __launch_bounds__(Cfg<Q>::NT, B200_DIAG_THREADS / Cfg<Q>::NT)
k_fused_diag(const __grid_constant__ DiagMats<P, Q> dm, const __grid_constant__ Material mt, int nelem,
             const int *__restrict__ offsets, const double *__restrict__ jcp, double *__restrict__ diag,
             double *__restrict__ evec) {
  constexpr int T = Cfg<Q>::T, EB = Cfg<Q>::EB, Q3 = Cfg<Q>::Q3, SE = Cfg<Q>::SE, P3 = P * P * P;
  constexpr int SY = Cfg<Q>::SY, SZ = Cfg<Q>::SZ, SC = Cfg<Q>::SC;
  constexpr int NC = JCache<PROB>::N;
  // selectors of term t = (d,d') per axis: (d == axis) + (d' == axis)
  constexpr int SELX[6] = {2, 0, 0, 0, 1, 1}, SELY[6] = {0, 2, 0, 1, 0, 1}, SELZ[6] = {0, 0, 2, 1, 1, 0};
  constexpr int VJ[6] = {0, 1, 2, 1, 0, 0}, VK[6] = {0, 1, 2, 2, 2, 1};
  extern __shared__ double smem[];
  const int tid = threadIdx.x;
  const int t = tid / EB, eb = tid - t * EB, a = t % Q, b = t / Q;
  const int blk = blockIdx.x;
  const int rem = nelem - blk * EB;
  const int ebn = FULL ? EB : (rem < EB ? rem : EB);   // FULL: compile-time plane strides (tail group: second launch)
  const bool act = t < T && (FULL || eb < ebn);
  const int e = blk * EB + eb;
  double *R = smem + eb * SE;  // 9 single-component lattices: terms 0..5, then the three z-selector sums
  const double *qlane = jcp + (size_t)blk * EB * NC * Q3 + (size_t)(FULL ? tid : t * ebn + eb);
  const size_t ebt = FULL ? (size_t)(EB * T) : (size_t)ebn * T;
  // the CTA's whole slab in one bulk L2 request: the first sweep then reads from L2 like the other two
  if (tid == 0) l2_prefetch_bulk(jcp + (size_t)blk * EB * NC * Q3, (unsigned)(ebt * Q * NC * sizeof(double)));

  // (M, kappa) of the thread's Q points, computed in the first sweep and kept in shared memory for the other two
  // components: private to the thread (same x-line owner in every sweep), [7][Q][lane] -> no barrier, no conflicts
  double *MK = smem + EB * SE + tid;
  constexpr int MKS = T * EB;  // lane stride
#pragma unroll 1
  for (int c = 0; c < 3; c++) {
    if (act) {
      double S[6][P];
#pragma unroll
      for (int tt = 0; tt < 6; tt++)
#pragma unroll
        for (int i = 0; i < P; i++) S[tt][i] = 0;
      if (c == 0) {
        double qn[NC];
#pragma unroll
        for (int n = 0; n < NC; n++) qn[n] = __ldg(qlane + (size_t)(n * Q) * ebt);
#pragma unroll 1
        for (int qx = 0; qx < Q; qx++) {
          double qd[NC], M[6], kappa;
#pragma unroll
          for (int n = 0; n < NC; n++) qd[n] = qn[n];
          if (qx + 1 < Q) {
#pragma unroll
            for (int n = 0; n < NC; n++) qn[n] = __ldg(qlane + (size_t)(n * Q + qx + 1) * ebt);
          }
          diag_blocks_point<PROB>(mt, qd, M, kappa);
#pragma unroll
          for (int tt = 0; tt < 6; tt++) MK[(tt * Q + qx) * MKS] = M[tt];
          MK[(6 * Q + qx) * MKS] = kappa;
          const double kc[3] = {qd[0], qd[3], qd[6]};
#pragma unroll
          for (int tt = 0; tt < 6; tt++) {
            double At = M[tt] + kappa * kc[VJ[tt]] * kc[VK[tt]];
            if (tt >= 3) At += At;
#pragma unroll
            for (int i = 0; i < P; i++) S[tt][i] += dm.M[SELX[tt]][qx * P + i] * At;
          }
        }
      } else {
        // K column c of every point of the line (L2 hits: the slab was read in the first sweep)
        double kq[Q][3];
#pragma unroll
        for (int qx = 0; qx < Q; qx++)
#pragma unroll
          for (int d = 0; d < 3; d++) kq[qx][d] = __ldg(qlane + (size_t)((3 * d + c) * Q + qx) * ebt);
#pragma unroll
        for (int qx = 0; qx < Q; qx++) {
          const double kappa = MK[(6 * Q + qx) * MKS];
#pragma unroll
          for (int tt = 0; tt < 6; tt++) {
            double At = MK[(tt * Q + qx) * MKS] + kappa * kq[qx][VJ[tt]] * kq[qx][VK[tt]];
            if (tt >= 3) At += At;
#pragma unroll
            for (int i = 0; i < P; i++) S[tt][i] += dm.M[SELX[tt]][qx * P + i] * At;
          }
        }
      }
#pragma unroll
      for (int tt = 0; tt < 6; tt++)
#pragma unroll
        for (int i = 0; i < P; i++) R[IDX(tt, i, a, b)] = S[tt][i];
    }
    __syncthreads();
    // y-lines (a = i < P, b = qz)
    if (act && a < P) {
      double Y[3][P];
#pragma unroll
      for (int s = 0; s < 3; s++)
#pragma unroll
        for (int j = 0; j < P; j++) Y[s][j] = 0;
#pragma unroll
      for (int tt = 0; tt < 6; tt++) {
        double in[Q];
#pragma unroll
        for (int qy = 0; qy < Q; qy++) in[qy] = R[IDX(tt, a, qy, b)];
#pragma unroll
        for (int j = 0; j < P; j++)
#pragma unroll
          for (int qy = 0; qy < Q; qy++) Y[SELZ[tt]][j] += dm.M[SELY[tt]][qy * P + j] * in[qy];
      }
#pragma unroll
      for (int s = 0; s < 3; s++)
#pragma unroll
        for (int j = 0; j < P; j++) R[IDX(6 + s, a, j, b)] = Y[s][j];
    }
    __syncthreads();
    // z-lines (a = i < P, b = j < P)
    if (act && a < P && b < P) {
      double acc[P];
#pragma unroll
      for (int k = 0; k < P; k++) acc[k] = 0;
#pragma unroll
      for (int s = 0; s < 3; s++) {
        double in[Q];
#pragma unroll
        for (int qz = 0; qz < Q; qz++) in[qz] = R[IDX(6 + s, a, b, qz)];
#pragma unroll
        for (int k = 0; k < P; k++)
#pragma unroll
          for (int qz = 0; qz < Q; qz++) acc[k] += dm.M[s][qz * P + k] * in[qz];
      }
      if (evec) {
#pragma unroll
        for (int k = 0; k < P; k++) evec[((size_t)e * P3 + (k * P + b) * P + a) * 3 + c] = acc[k];
      } else {
#pragma unroll
        for (int k = 0; k < P; k++) {
          const int o = __ldg(offsets + (size_t)e * P3 + (k * P + b) * P + a);
          atomicAdd(diag + o + c, acc[k]);
        }
      }
    }
    // the next component's x-stage writes lattices 0..5 (their readers passed the second barrier) and its
    // y-stage writes 6..8 only behind the next barrier, which no thread reaches before finishing this z-stage
  }
}

// -----------------------------------------------------------------------------------
// p-multigrid transfer: out_L += Eo^T I^(T) Ei in_L  (matops.c:115-203)
// PC nodes -> PF nodes with the interpolation matrix J [PF][PC]; same line machinery.
// -----------------------------------------------------------------------------------
template <int PC, int PF> struct XferMats { double J[PF * PC]; };

// Shared memory of the transfer kernel: two lattices of three components per element (6 SC), element stride padded
// like Cfg<Q>::SE.  The L-vector is touched only by two flat sweeps in L-vector order, f = (element, node, component)
// with the component fastest: consecutive lanes read / write consecutive interlaced dofs, so a warp's request covers
// a few full sectors instead of 32 separate ones (the line owners of one warp belong to EB different elements).
__host__ __device__ constexpr int xfer_se(int Q) {
  return elems_per_block(Q) == 16 ? ((6 * apply_sc(Q, Q)) | 1)
                                  : 6 * apply_sc(Q, Q) + ((16 / elems_per_block(Q) - (6 * apply_sc(Q, Q)) % 16) + 16) % 16;
}

#ifndef B200_XFER_LINE_IO
// resident CTAs per SM asked of the compiler (measured, profiles/r2_transfer_ab.txt): the prolongation (few loads,
// many stores) gains from 8 (64 registers at PF = 5); the restriction onto PF = 5 keeps its 12 offset -> value ->
// multiplicity load chains in flight only with the default allocation (a 64-register cap spills), below that 8 wins
#ifndef B200_XFER_MIN_CTAS_PROLONG
#define B200_XFER_MIN_CTAS_PROLONG 8
#endif
#ifndef B200_XFER_MIN_CTAS_RESTRICT
#define B200_XFER_MIN_CTAS_RESTRICT(PF) ((PF) <= 3 ? 8 : 1)
#endif
template <int PC, int PF, int TR>
__global__ void __launch_bounds__(Cfg<PF>::NT, TR ? B200_XFER_MIN_CTAS_RESTRICT(PF) : B200_XFER_MIN_CTAS_PROLONG)
k_transfer(const __grid_constant__ XferMats<PC, PF> m, int nelem, const int *__restrict__ offc,
           const int *__restrict__ offf, const double *__restrict__ mult, int inject, const double *__restrict__ in,
           double *__restrict__ out, double *__restrict__ evec, const unsigned short *__restrict__ gtab) {
  constexpr int Q = PF;  // lattice extent used for smem indexing
  constexpr int T = Cfg<Q>::T, EB = Cfg<Q>::EB, NT = Cfg<Q>::NT, SE = xfer_se(Q);
  constexpr int SY = Cfg<Q>::SY, SZ = Cfg<Q>::SZ, SC = Cfg<Q>::SC;
  constexpr int NI = TR ? PF : PC, NO = TR ? PC : PF;  // line extents in / out
  constexpr int NI3 = NI * NI * NI, NO3 = NO * NO * NO;
  static_assert(3 * NO3 <= 3 * SC, "interlaced nodal output must fit in the first lattice triple");
  extern __shared__ double smem[];
  const int tid = threadIdx.x, blk = blockIdx.x;
  const int t = tid / EB, eb = tid - t * EB, a = t % Q, b = t / Q;
  const int rem = nelem - blk * EB;
  const int ebn = rem < EB ? rem : EB;
  const bool act = t < T && eb < ebn;
  double *R0 = smem + eb * SE, *R1 = R0 + 3 * SC;
#define JM(o, i) (TR ? m.J[(i) * PC + (o)] : m.J[(o) * PC + (i)])
  // ---- gather sweep: input nodes of the CTA's elements in L-vector order -> lattice R1 of each element
  {
    constexpr int NIT = (EB * 3 * NI3 + NT - 1) / NT;
    const int total = ebn * 3 * NI3;
    const int *oin = (TR ? offf : offc) + (size_t)blk * EB * NI3;
    // every load is unconditional (index clamped into the CTA's range) so that the NIT dependent pairs
    // offset -> value are all in flight together; only the shared-memory store is predicated
    // the lattice word of each f is the same for every CTA: a small table instead of five divisions per entry
    double v[NIT];
    int o[NIT];
    unsigned short w[NIT];
#pragma unroll
    for (int it = 0; it < NIT; it++) {
      const int f = tid + it * NT, fc = f < total ? f : total - 1;
      const int node = fc / 3;  // runs over (element, node of the element)
      o[it] = __ldg(oin + node) + (fc - node * 3);
      w[it] = __ldg(gtab + fc);
    }
#pragma unroll
    for (int it = 0; it < NIT; it++) v[it] = __ldg(in + o[it]);
    if (TR && mult) {
#pragma unroll
      for (int it = 0; it < NIT; it++) v[it] *= __ldg(mult + o[it]);
    }
#pragma unroll
    for (int it = 0; it < NIT; it++) {
      const int f = tid + it * NT;
      if (f < total) smem[w[it]] = v[it];
    }
  }
  __syncthreads();
  // ---- z-lines (a = i, b = j): contract z
  if (act && a < NI && b < NI) {
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double l[NI];
#pragma unroll
      for (int k = 0; k < NI; k++) l[k] = R1[IDX(c, a, b, k)];
#pragma unroll
      for (int z = 0; z < NO; z++) {
        double s = 0;
#pragma unroll
        for (int k = 0; k < NI; k++) s += JM(z, k) * l[k];
        R0[IDX(c, a, b, z)] = s;
      }
    }
  }
  __syncthreads();
  // ---- y-lines (a = i < NI, b = z < NO)
  if (act && a < NI && b < NO) {
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double l[NI];
#pragma unroll
      for (int j = 0; j < NI; j++) l[j] = R0[IDX(c, a, j, b)];
#pragma unroll
      for (int yy = 0; yy < NO; yy++) {
        double s = 0;
#pragma unroll
        for (int j = 0; j < NI; j++) s += JM(yy, j) * l[j];
        R1[IDX(c, a, yy, b)] = s;
      }
    }
  }
  __syncthreads();
  // ---- x-lines (a = y < NO, b = z < NO) -> nodal output, interlaced [node][component], over lattice R0 (free now)
  if (act && a < NO && b < NO) {
    double *Rn = R0 + ((b * NO + a) * NO) * 3;
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double l[NI];
#pragma unroll
      for (int i = 0; i < NI; i++) l[i] = R1[IDX(c, i, a, b)];
#pragma unroll
      for (int xx = 0; xx < NO; xx++) {
        double s = 0;
#pragma unroll
        for (int i = 0; i < NI; i++) s += JM(xx, i) * l[i];
        Rn[xx * 3 + c] = s;
      }
    }
  }
  __syncthreads();
  // ---- scatter sweep in L-vector order
  {
    constexpr int NIT = (EB * 3 * NO3 + NT - 1) / NT;
    const int total = ebn * 3 * NO3;
    const int *oout = (TR ? offc : offf) + (size_t)blk * EB * NO3;
    double val[NIT];
    int dst[NIT];
#pragma unroll
    for (int it = 0; it < NIT; it++) {  // unconditional loads (clamped), predicated stores: see the gather sweep
      const int f = tid + it * NT, fc = f < total ? f : total - 1;
      const int el = fc / (3 * NO3), node = fc / 3;
      val[it] = smem[el * SE + (fc - el * 3 * NO3)];
      dst[it] = __ldg(oout + node) + (fc - node * 3);
    }
    // inject: the elements sharing a node store the same interpolant there, bit for bit when they share their local
    // axes; a differently oriented neighbour contracts in another order and may differ in the last bit
    if (!TR && inject) {
#pragma unroll
      for (int it = 0; it < NIT; it++)
        if (tid + it * NT < total) out[dst[it]] = val[it];
      return;
    }
    if (!TR && mult) {
#pragma unroll
      for (int it = 0; it < NIT; it++)
        if (tid + it * NT < total) val[it] *= __ldg(mult + dst[it]);
    }
    if (evec) {  // deterministic mode: element outputs [e][node][comp], summed in a fixed order by the caller
      double *ev = evec + (size_t)blk * EB * 3 * NO3;
#pragma unroll
      for (int it = 0; it < NIT; it++)
        if (tid + it * NT < total) ev[tid + it * NT] = val[it];
    } else {
#pragma unroll
      for (int it = 0; it < NIT; it++)
        if (tid + it * NT < total) atomicAdd(out + dst[it], val[it]);
    }
  }
#undef JM
}
#else  // B200_XFER_LINE_IO: the round-1 form, every line owner gathers and scatters its own nodes
template <int PC, int PF, int TR>
__global__ void __launch_bounds__(Cfg<PF>::NT)
k_transfer(const __grid_constant__ XferMats<PC, PF> m, int nelem, const int *__restrict__ offc,
           const int *__restrict__ offf, const double *__restrict__ mult, int inject, const double *__restrict__ in,
           double *__restrict__ out, double *__restrict__ evec, const unsigned short *__restrict__) {
  constexpr int Q = PF;  // lattice extent used for smem indexing
  constexpr int T = Cfg<Q>::T, EB = Cfg<Q>::EB, SE = Cfg<Q>::SE;
  constexpr int SY = Cfg<Q>::SY, SZ = Cfg<Q>::SZ, SC = Cfg<Q>::SC;
  constexpr int NI = TR ? PF : PC, NO = TR ? PC : PF;  // line extents in / out
  extern __shared__ double smem[];
  const int tid = threadIdx.x;
  const int t = tid / EB, eb = tid - t * EB, a = t % Q, b = t / Q;
  const int rem = nelem - blockIdx.x * EB;
  const int ebn = rem < EB ? rem : EB;
  const bool act = t < T && eb < ebn;
  const int e = blockIdx.x * EB + eb;
  double *R0 = smem + eb * SE, *R1 = R0 + 3 * SC;
  const int *oin = (TR ? offf : offc) + (size_t)e * NI * NI * NI;
  const int *oout = (TR ? offc : offf) + (size_t)e * NO * NO * NO;
#define JM(o, i) (TR ? m.J[(i) * PC + (o)] : m.J[(o) * PC + (i)])
  // z-lines (a = i, b = j) gather + contract z
  if (act && a < NI && b < NI) {
    double r[3][NI];
#pragma unroll
    for (int k = 0; k < NI; k++) {
      const int o = __ldg(oin + (k * NI + b) * NI + a);
#pragma unroll
      for (int c = 0; c < 3; c++) {
        double v = __ldg(in + o + c);
        if (TR && mult) v *= __ldg(mult + o + c);
        r[c][k] = v;
      }
    }
#pragma unroll
    for (int c = 0; c < 3; c++)
#pragma unroll
      for (int z = 0; z < NO; z++) {
        double s = 0;
#pragma unroll
        for (int k = 0; k < NI; k++) s += JM(z, k) * r[c][k];
        R0[IDX(c, a, b, z)] = s;
      }
  }
  __syncthreads();
  // y-lines (a = i < NI, b = z < NO)
  if (act && a < NI && b < NO) {
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double l[NI];
#pragma unroll
      for (int j = 0; j < NI; j++) l[j] = R0[IDX(c, a, j, b)];
#pragma unroll
      for (int yy = 0; yy < NO; yy++) {
        double s = 0;
#pragma unroll
        for (int j = 0; j < NI; j++) s += JM(yy, j) * l[j];
        R1[IDX(c, a, yy, b)] = s;
      }
    }
  }
  __syncthreads();
  // x-lines (a = y < NO, b = z < NO), scatter
  if (act && a < NO && b < NO) {
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double l[NI];
#pragma unroll
      for (int i = 0; i < NI; i++) l[i] = R1[IDX(c, i, a, b)];
#pragma unroll
      for (int xx = 0; xx < NO; xx++) {
        double s = 0;
#pragma unroll
        for (int i = 0; i < NI; i++) s += JM(xx, i) * l[i];
        const int o = __ldg(oout + (b * NO + a) * NO + xx);
        if (!TR && inject) {  // same interpolant at every holder up to the last bit (see the default form above)
          out[o + c] = s;
          continue;
        }
        if (!TR && mult) s *= __ldg(mult + o + c);
        if (evec) evec[((size_t)e * NO * NO * NO + (b * NO + a) * NO + xx) * 3 + c] = s;
        else atomicAdd(out + o + c, s);
      }
    }
  }
#undef JM
}

#endif  // B200_XFER_LINE_IO

// -----------------------------------------------------------------------------------
// host side
// -----------------------------------------------------------------------------------

// Gc = D * pinv(B): the unique-on-range(B) matrix with Gc B = D (P <= Q, B full column rank).
static int collocated_grad(int P, int Q, const double *B, const double *D, double *Gc) {
  double N[8 * 8], Ninv[8 * 8], tmp[8 * 8];
  for (int i = 0; i < P; i++)
    for (int j = 0; j < P; j++) {
      double s = 0;
      for (int q = 0; q < Q; q++) s += B[q * P + i] * B[q * P + j];
      N[i * P + j] = s;
      Ninv[i * P + j] = i == j ? 1.0 : 0.0;
    }
  for (int col = 0; col < P; col++) {  // Gauss-Jordan with partial pivoting
    int piv = col;
    for (int r = col + 1; r < P; r++)
      if (fabs(N[r * P + col]) > fabs(N[piv * P + col])) piv = r;
    if (fabs(N[piv * P + col]) < 1e-300) return 1;
    if (piv != col)
      for (int j = 0; j < P; j++) {
        double t = N[col * P + j]; N[col * P + j] = N[piv * P + j]; N[piv * P + j] = t;
        t = Ninv[col * P + j]; Ninv[col * P + j] = Ninv[piv * P + j]; Ninv[piv * P + j] = t;
      }
    const double d = 1.0 / N[col * P + col];
    for (int j = 0; j < P; j++) { N[col * P + j] *= d; Ninv[col * P + j] *= d; }
    for (int r = 0; r < P; r++)
      if (r != col) {
        const double f = N[r * P + col];
        for (int j = 0; j < P; j++) { N[r * P + j] -= f * N[col * P + j]; Ninv[r * P + j] -= f * Ninv[col * P + j]; }
      }
  }
  // tmp = D * Ninv  [Q][P];  Gc = tmp * B^T  [Q][Q]
  for (int q = 0; q < Q; q++)
    for (int j = 0; j < P; j++) {
      double s = 0;
      for (int i = 0; i < P; i++) s += D[q * P + i] * Ninv[i * P + j];
      tmp[q * P + j] = s;
    }
  for (int q = 0; q < Q; q++)
    for (int r = 0; r < Q; r++) {
      double s = 0;
      for (int j = 0; j < P; j++) s += tmp[q * P + j] * B[r * P + j];
      Gc[q * Q + r] = s;
    }
  // one step of iterative refinement is unnecessary at these sizes; verify instead
  double err = 0, nrm = 0;
  for (int q = 0; q < Q; q++)
    for (int i = 0; i < P; i++) {
      double s = 0;
      for (int r = 0; r < Q; r++) s += Gc[q * Q + r] * B[r * P + i];
      err = fmax(err, fabs(s - D[q * P + i]));
      nrm = fmax(nrm, fabs(D[q * P + i]));
    }
  return err <= 1e-12 * nrm ? 0 : 2;
}

// the same for the generated fused kernels of user QFunctions (b200_jit.cu)
int collocated_grad_1d(int P, int Q, const double *B, const double *D, double *Gc) { return collocated_grad(P, Q, B, D, Gc); }

template <typename K> static int opt_in_smem(K kern, size_t bytes) {
  if (bytes > 48 * 1024) B200_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return 0;
}

// per-device one-time state of a kernel instantiation (opt-in shared memory size, small device tables):
// one process may drive several devices (CeedInit "/gpu/b200:device_id=N")
constexpr int MAX_DEVICES = 64;
struct PerDevice {
  bool configured[MAX_DEVICES] = {};
  void *table[MAX_DEVICES] = {};
};
static int current_device(int *dev) {
  B200_CHECK(cudaGetDevice(dev));
  if (*dev < 0 || *dev >= MAX_DEVICES) return set_error_msg("device ordinal out of range");
  return 0;
}

// the collocated derivative of a basis is computed once per (P, Q) instantiation and reused while the caller
// keeps passing the same interp1d / grad1d values
template <int P, int Q> static int cached_mats(const double *hB, const double *hD, Mats<P, Q> &m) {
  static Mats<P, Q> cache;
  static double keyB[Q * P], keyD[Q * P];
  static bool valid = false;
  if (!valid || memcmp(keyB, hB, sizeof keyB) || memcmp(keyD, hD, sizeof keyD)) {
    for (int i = 0; i < Q * P; i++) cache.B[i] = hB[i];
    if (collocated_grad(P, Q, hB, hD, cache.Gc)) {
      valid = false;
      return set_error_msg("basis: no collocated gradient with Gc*B = D (rank-deficient interp1d)");
    }
    memcpy(keyB, hB, sizeof keyB);
    memcpy(keyD, hD, sizeof keyD);
    valid = true;
  }
  m = cache;
  return 0;
}

// one wave of resident CTAs (5 per SM on 148 SMs), rounded up: how far ahead a CTA prefetches element offsets
constexpr int OFFSETS_AHEAD = 1024;
// how many groups ahead a CTA prefetches the L-vector entries of a later gather (0 = off; must stay below OFFSETS_AHEAD)
constexpr int X_AHEAD = 0;
// how many groups ahead a CTA requests the per-point slab (0 = its own)
constexpr int SLAB_AHEAD = 0;

template <int P, int Q, int PROB, int MODE>
static int launch_apply(const Material &mt, int nelem, const double *hB, const double *hD, const int *offsets,
                        const double *qa, double *gradu, const double *x, double *y, double *evec) {
  Mats<P, Q> m;
  if (int rc = cached_mats<P, Q>(hB, hD, m)) return rc;
  auto kern = k_fused_apply<P, Q, PROB, MODE, true>;
  auto kern_tail = k_fused_apply<P, Q, PROB, MODE, false>;
  constexpr int EB = Cfg<Q>::EB, P3 = P * P * P, SC = apply_sc(P, Q), SE = apply_se(Q, SC);
  constexpr int NC = MODE == MODE_JACOBIAN ? JCache<PROB>::N : 10, Q3 = Q * Q * Q;
  const size_t smem_bytes = sizeof(double) * EB * SE + sizeof(int) * EB * P3;
  static PerDevice pd;
  int dev;
  if (int rc = current_device(&dev)) return rc;
  if (!pd.configured[dev]) {
    if (int rc = opt_in_smem(kern, smem_bytes)) return rc;
    if (int rc = opt_in_smem(kern_tail, smem_bytes)) return rc;
    // scatter table: f = (el, node, c) with c fastest -> shared-memory word | offset index << 16 | c << 28
    static_assert(EB * SE < 65536 && EB * P3 < 4096, "scatter table packing");
    unsigned h[EB * P3 * 3];
    for (int el = 0; el < EB; el++)
      for (int node = 0; node < P3; node++)
        for (int c = 0; c < 3; c++) {
          h[(el * P3 + node) * 3 + c] = (unsigned)(el * SE + node * 3 + c) | ((unsigned)(el * P3 + node) << 16) | ((unsigned)c << 28);
        }
    B200_CHECK(cudaMalloc(&pd.table[dev], sizeof h));
    B200_CHECK(cudaMemcpy(pd.table[dev], h, sizeof h, cudaMemcpyHostToDevice));
    pd.configured[dev] = true;
  }
  const unsigned *d_tab = static_cast<const unsigned *>(pd.table[dev]);
#ifdef B200_NO_FULL
  if (nelem) {
    kern_tail<<<(nelem + EB - 1) / EB, Cfg<Q>::NT, smem_bytes, g_stream>>>(m, mt, nelem, offsets, qa, gradu, x, y, d_tab, 0, evec, 0, 0);
    B200_LAUNCH_CHECK("k_fused_apply");
    return 0;
  }
#endif
  static const int ahead = getenv("B200_OFFSETS_AHEAD") ? atoi(getenv("B200_OFFSETS_AHEAD")) : OFFSETS_AHEAD;
  static const int xahead = getenv("B200_X_AHEAD") ? atoi(getenv("B200_X_AHEAD")) : X_AHEAD;
  static const int sahead = getenv("B200_SLAB_AHEAD") ? atoi(getenv("B200_SLAB_AHEAD")) : SLAB_AHEAD;
  const int nfull = nelem / EB, ntail = nelem - nfull * EB;
  if (nfull) {
    kern<<<nfull, Cfg<Q>::NT, smem_bytes, g_stream>>>(m, mt, nfull * EB, offsets, qa, gradu, x, y, d_tab, ahead, evec, xahead, sahead);
    B200_LAUNCH_CHECK("k_fused_apply");
  }
  if (ntail) {  // the partial group at the end of the element range: same kernel with run-time group extent
    const size_t e0 = (size_t)nfull * EB;
    kern_tail<<<1, Cfg<Q>::NT, smem_bytes, g_stream>>>(m, mt, ntail, offsets + e0 * P3, qa + e0 * NC * Q3,
                                                       gradu ? gradu + e0 * 9 * Q3 : nullptr, x, y, d_tab, 0,
                                                       evec ? evec + e0 * 3 * P3 : nullptr, 0, 0);
    B200_LAUNCH_CHECK("k_fused_apply(tail)");
  }
  return 0;
}

template <int P, int Q, int PROB>
static int launch_diag(const Material &mt, int nelem, const double *hB, const double *hD, const int *offsets,
                       const double *jc, double *diag, double *evec) {
  DiagMats<P, Q> dm;
  for (int i = 0; i < Q * P; i++) {
    dm.M[0][i] = hB[i] * hB[i];
    dm.M[1][i] = hB[i] * hD[i];
    dm.M[2][i] = hD[i] * hD[i];
  }
  auto kern = k_fused_diag<P, Q, PROB, true>;
  auto kern_tail = k_fused_diag<P, Q, PROB, false>;
  // nine lattices per element + the per-thread (M, kappa) store of the first sweep
  constexpr size_t diag_smem = Cfg<Q>::SMEM + sizeof(double) * 7 * Q * Cfg<Q>::T * Cfg<Q>::EB;
  constexpr int EB = Cfg<Q>::EB, P3 = P * P * P, Q3 = Q * Q * Q, NC = JCache<PROB>::N;
  static PerDevice pd;
  int dev;
  if (int rc = current_device(&dev)) return rc;
  if (!pd.configured[dev]) {
    if (int rc = opt_in_smem(kern, diag_smem)) return rc;
    if (int rc = opt_in_smem(kern_tail, diag_smem)) return rc;
    pd.configured[dev] = true;
  }
  const int nfull = nelem / EB, ntail = nelem - nfull * EB;
  if (nfull) {
    kern<<<nfull, Cfg<Q>::NT, diag_smem, g_stream>>>(dm, mt, nfull * EB, offsets, jc, diag, evec);
    B200_LAUNCH_CHECK("k_fused_diag");
  }
  if (ntail) {
    const size_t e0 = (size_t)nfull * EB;
    kern_tail<<<1, Cfg<Q>::NT, diag_smem, g_stream>>>(dm, mt, ntail, offsets + e0 * P3, jc + e0 * NC * Q3, diag,
                                                      evec ? evec + e0 * 3 * P3 : nullptr);
    B200_LAUNCH_CHECK("k_fused_diag(tail)");
  }
  return 0;
}

template <int PC, int PF, int TR>
static int launch_transfer(int nelem, const double *hJ, const int *offc, const int *offf, const double *mult, int inject,
                           const double *in, double *out, double *evec) {
  XferMats<PC, PF> m;
  for (int i = 0; i < PF * PC; i++) m.J[i] = hJ[i];
  auto kern = k_transfer<PC, PF, TR>;
#ifndef B200_XFER_LINE_IO
  constexpr size_t xfer_smem = (size_t)Cfg<PF>::EB * xfer_se(PF) * sizeof(double);
#else
  constexpr size_t xfer_smem = Cfg<PF>::SMEM;
#endif
  static PerDevice pd;
  int dev;
  if (int rc = current_device(&dev)) return rc;
  if (!pd.configured[dev]) {
    if (int rc = opt_in_smem(kern, xfer_smem)) return rc;
    // gather table: f = (el, node, c) with c fastest -> shared-memory word of lattice R1 of element el
    constexpr int EB = Cfg<PF>::EB, NI = TR ? PF : PC, SC = Cfg<PF>::SC, SY = Cfg<PF>::SY, SZ = Cfg<PF>::SZ;
    static_assert(EB * xfer_se(PF) < 65536, "gather table packing");
    unsigned short h[EB * NI * NI * NI * 3];
    for (int el = 0; el < EB; el++)
      for (int z = 0; z < NI; z++)
        for (int y = 0; y < NI; y++)
          for (int x = 0; x < NI; x++)
            for (int c = 0; c < 3; c++)
              h[((el * NI * NI * NI) + (z * NI + y) * NI + x) * 3 + c] = (unsigned short)(el * xfer_se(PF) + 3 * SC + IDX(c, x, y, z));
    B200_CHECK(cudaMalloc(&pd.table[dev], sizeof h));
    B200_CHECK(cudaMemcpy(pd.table[dev], h, sizeof h, cudaMemcpyHostToDevice));
    pd.configured[dev] = true;
  }
  const int nblk = (nelem + Cfg<PF>::EB - 1) / Cfg<PF>::EB;
  if (nblk == 0) return 0;
  kern<<<nblk, Cfg<PF>::NT, xfer_smem, g_stream>>>(m, nelem, offc, offf, mult, inject, in, out, evec,
                                                    static_cast<const unsigned short *>(pd.table[dev]));
  B200_LAUNCH_CHECK("k_transfer");
  return 0;
}

// (P, Q) pairs instantiated: every level of p-MG hierarchies up to degree 4 (Q <= 5); anything
// else runs through the generic restriction/basis/QFunction kernels
#define B200_FOR_PQ(X) \
  X(2, 2) X(2, 3) X(3, 3) X(2, 4) X(3, 4) X(4, 4) X(2, 5) X(3, 5) X(4, 5) X(5, 5)

template <int PROB, int MODE>
static int dispatch_apply(int P, int Q, const Material &mt, int nelem, const double *hB, const double *hD,
                          const int *offsets, const double *qa, double *gradu, const double *x, double *y, double *evec) {
#define X(p, q) \
  if (P == p && Q == q) return launch_apply<p, q, PROB, MODE>(mt, nelem, hB, hD, offsets, qa, gradu, x, y, evec);
  B200_FOR_PQ(X)
#undef X
  return set_error_msg("fused apply: (P,Q) not instantiated");
}

template <int PROB>
static int dispatch_diag(int P, int Q, const Material &mt, int nelem, const double *hB, const double *hD,
                         const int *offsets, const double *jc, double *diag, double *evec) {
#define X(p, q) \
  if (P == p && Q == q) return launch_diag<p, q, PROB>(mt, nelem, hB, hD, offsets, jc, diag, evec);
  B200_FOR_PQ(X)
#undef X
  return set_error_msg("fused diagonal: (P,Q) not instantiated");
}

}  // namespace b200

using namespace b200;

extern "C" int b200_fused_supported(int P, int Q) {
#define X(p, q) \
  if (P == p && Q == q) return 1;
  B200_FOR_PQ(X)
#undef X
  return 0;
}

// shared-memory lattice strides of the fused apply kernel for (P, Q): out = {SY, SZ, SC, SE, EB, NT}
extern "C" int b200_apply_smem_layout(int P, int Q, int *out) {
#define X(p, q)                                                                                   \
  if (P == p && Q == q) {                                                                         \
    out[0] = Cfg<q>::SY; out[1] = Cfg<q>::SZ; out[2] = apply_sc(p, q); out[3] = apply_se(q, apply_sc(p, q)); \
    out[4] = Cfg<q>::EB; out[5] = Cfg<q>::NT;                                                     \
    return 0;                                                                                     \
  }
  B200_FOR_PQ(X)
#undef X
  return set_error_msg("b200_apply_smem_layout: (P,Q) not instantiated");
}

extern "C" int b200_jcache_ncomp(int problem) {
  return problem == B200_PROB_LINELAS ? 9 : problem == B200_PROB_HYPERSS ? 10 : problem == B200_PROB_HYPERFS ? 16 : -1;
}

extern "C" int b200_apply_residual(int problem, const b200_physics *phys, int nelem, int P, int Q,
                                   const double *hB, const double *hD, const int *d_offsets,
                                   const double *d_qdata, double *d_gradu, const double *d_x, double *d_y, double *d_evec) {
  const Material mt = make_material(phys);
  switch (problem) {
    case B200_PROB_LINELAS: return dispatch_apply<B200_PROB_LINELAS, MODE_RESIDUAL>(P, Q, mt, nelem, hB, hD, d_offsets, d_qdata, d_gradu, d_x, d_y, d_evec);
    case B200_PROB_HYPERSS: return dispatch_apply<B200_PROB_HYPERSS, MODE_RESIDUAL>(P, Q, mt, nelem, hB, hD, d_offsets, d_qdata, d_gradu, d_x, d_y, d_evec);
    case B200_PROB_HYPERFS: return dispatch_apply<B200_PROB_HYPERFS, MODE_RESIDUAL>(P, Q, mt, nelem, hB, hD, d_offsets, d_qdata, d_gradu, d_x, d_y, d_evec);
  }
  return set_error_msg("b200_apply_residual: unknown problem");
}

extern "C" int b200_apply_jacobian(int problem, const b200_physics *phys, int nelem, int P, int Q,
                                   const double *hB, const double *hD, const int *d_offsets,
                                   const double *d_jcache, const double *d_x, double *d_y, double *d_evec) {
  const Material mt = make_material(phys);
  switch (problem) {
    case B200_PROB_LINELAS: return dispatch_apply<B200_PROB_LINELAS, MODE_JACOBIAN>(P, Q, mt, nelem, hB, hD, d_offsets, d_jcache, nullptr, d_x, d_y, d_evec);
    case B200_PROB_HYPERSS: return dispatch_apply<B200_PROB_HYPERSS, MODE_JACOBIAN>(P, Q, mt, nelem, hB, hD, d_offsets, d_jcache, nullptr, d_x, d_y, d_evec);
    case B200_PROB_HYPERFS: return dispatch_apply<B200_PROB_HYPERFS, MODE_JACOBIAN>(P, Q, mt, nelem, hB, hD, d_offsets, d_jcache, nullptr, d_x, d_y, d_evec);
  }
  return set_error_msg("b200_apply_jacobian: unknown problem");
}

extern "C" int b200_apply_diagonal(int problem, const b200_physics *phys, int nelem, int P, int Q,
                                   const double *hB, const double *hD, const int *d_offsets,
                                   const double *d_jcache, double *d_diag, double *d_evec) {
  const Material mt = make_material(phys);
  switch (problem) {
    case B200_PROB_LINELAS: return dispatch_diag<B200_PROB_LINELAS>(P, Q, mt, nelem, hB, hD, d_offsets, d_jcache, d_diag, d_evec);
    case B200_PROB_HYPERSS: return dispatch_diag<B200_PROB_HYPERSS>(P, Q, mt, nelem, hB, hD, d_offsets, d_jcache, d_diag, d_evec);
    case B200_PROB_HYPERFS: return dispatch_diag<B200_PROB_HYPERFS>(P, Q, mt, nelem, hB, hD, d_offsets, d_jcache, d_diag, d_evec);
  }
  return set_error_msg("b200_apply_diagonal: unknown problem");
}

extern "C" int b200_jcache_build(int problem, int nelem, int Q, const double *d_qdata, const double *d_gradu,
                                 double *d_jcache) {
  if (Q < 2 || Q > 8) return set_error_msg("b200_jcache_build: Q out of range");
  if (nelem == 0) return 0;
  const size_t npts = (size_t)nelem * Q * Q * Q;
  const int nt = 256;
  size_t nb = (npts + nt - 1) / nt;
  if (nb > 148 * 64) nb = 148 * 64;
  switch (problem) {
    case B200_PROB_LINELAS: k_jcache_build<B200_PROB_LINELAS><<<(int)nb, nt, 0, g_stream>>>(nelem, Q, d_qdata, d_gradu, d_jcache); break;
    case B200_PROB_HYPERSS: k_jcache_build<B200_PROB_HYPERSS><<<(int)nb, nt, 0, g_stream>>>(nelem, Q, d_qdata, d_gradu, d_jcache); break;
    case B200_PROB_HYPERFS: k_jcache_build<B200_PROB_HYPERFS><<<(int)nb, nt, 0, g_stream>>>(nelem, Q, d_qdata, d_gradu, d_jcache); break;
    default: return set_error_msg("b200_jcache_build: unknown problem");
  }
  B200_LAUNCH_CHECK("k_jcache_build");
  return 0;
}

extern "C" int b200_apply_transfer(int transpose, int nelem, int Pc, int Pf, const double *hJ, const int *d_offc,
                                   const int *d_offf, const double *d_mult, int inject, const double *d_in, double *d_out,
                                   double *d_evec) {
  if (inject && (transpose || !d_mult)) return set_error_msg("b200_apply_transfer: inject is the prolongation with multiplicity scaling");
#define XF(pc, pf)                                                                                                      \
  if (Pc == pc && Pf == pf)                                                                                             \
    return transpose ? launch_transfer<pc, pf, 1>(nelem, hJ, d_offc, d_offf, d_mult, 0, d_in, d_out, d_evec)            \
                     : launch_transfer<pc, pf, 0>(nelem, hJ, d_offc, d_offf, d_mult, inject, d_in, d_out, d_evec);
  XF(2, 3) XF(3, 4) XF(4, 5) XF(3, 5) XF(2, 4) XF(2, 5)
#undef XF
  return set_error_msg("b200_apply_transfer: (Pc,Pf) not instantiated");
}
