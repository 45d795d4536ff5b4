// K12: the fused operator kernel around a user QFunction compiled at run time ("/gpu/b200:jit").
//
// Device-only template.  It is not compiled into the library: the build embeds it as a string (b200_jit.cu), and NVRTC
// compiles it together with the user's program and a generated prefix that defines, before this text:
//   B200_K12_P, B200_K12_Q                       the basis (P, Q), one of B200_FOR_PQ
//   B200_K12_SY, _SZ, _SC, _SE, _EB, _NT         the shared-memory lattice of b200_apply_smem_layout(P, Q)
//   b200_jit_ctx_t, b200_k12_fields_t            the context bytes and the field pointers (by QFunction field index)
//   b200_k12_point(ctx, f, grp, pos, cs, H, W, padd)
//       one call of the user function with Q = 1 at one point: the active input in[d*3 + c] = H[c][d], the passive
//       inputs loaded from their q-blocked slabs (field i at f.in[i] + grp * size_i + pos + comp * cs), the active
//       output out[k*3 + c] returned as W[c][k], the passive outputs stored (padd = 0) or added (padd != 0) the same way
// and, after it, the two extern "C" kernels that call b200_k12_body<true> (full groups) and <false> (the tail group).
//
// The stages are those of k_fused_apply (b200_fused.cu): offsets gather along z-lines, the sum-factorised gradient
// along the three line orientations (interpolation B, then the collocated derivative Gc with Gc B = D), the point
// function at the Q points of each x-line, the exact transposed stages, and the scatter-add (FP64 atomics, or plain
// stores to an E-vector [e][node][comp] that the caller sums in a fixed order).  The two kernels share the lattice
// layout, not the code: the built-in kernel's register caps, look-ahead loads and scatter table are tuned to the
// built-in point functions.
#ifndef B200_JIT_FUSED_CUH
#define B200_JIT_FUSED_CUH

struct b200_k12_mats_t {
  double B[B200_K12_Q * B200_K12_P];   // interp1d [Q][P]
  double Gc[B200_K12_Q * B200_K12_Q];  // collocated derivative at the quadrature points
};

#define B200_K12_IDX(c, x, y, z) ((c) * SC + (z) * SZ + (y) * SY + (x))

template <bool FULL>
__device__ __forceinline__ void b200_k12_body(const b200_k12_mats_t &m, const b200_jit_ctx_t &ctx,
                                              const b200_k12_fields_t &f, const int nelem, const int *__restrict__ offsets,
                                              const double *__restrict__ x, double *__restrict__ y,
                                              double *__restrict__ evec, const int padd) {
  constexpr int P = B200_K12_P, Q = B200_K12_Q, T = Q * Q, Q3 = Q * Q * Q, P3 = P * P * P;
  constexpr int SY = B200_K12_SY, SZ = B200_K12_SZ, SC = B200_K12_SC, SE = B200_K12_SE, EB = B200_K12_EB;
  constexpr int NT = B200_K12_NT;
  static_assert(3 * P3 <= 6 * SC, "interlaced nodal output must fit in the first two lattices");
  extern __shared__ double smem[];
  const int tid = threadIdx.x;
  const int t = tid / EB, eb = tid - t * EB, a = t % Q, b = t / Q;
  const int blk = blockIdx.x;
  const int rem = nelem - blk * EB;
  const int ebn = FULL ? EB : (rem < EB ? rem : EB);
  const bool act = t < T && (FULL || eb < ebn);
  const int e = blk * EB + eb;
  double *R0 = smem + eb * SE, *R1 = R0 + 3 * SC, *R2 = R1 + 3 * SC;
  int *soff = reinterpret_cast<int *>(smem + EB * SE);
  // q-blocked slabs of the passive fields: group base (per component), this lane, the plane stride
  const size_t grp = (size_t)blk * EB * Q3;
  const size_t ebt = FULL ? (size_t)(EB * T) : (size_t)ebn * T;
  const size_t lane = FULL ? (size_t)tid : (size_t)(t * ebn + eb);

  // ---- gather node z-lines, contract z with B
  if (act && a < P && b < P) {
    double r[3][P];
    const int *off = offsets + (size_t)e * P3 + b * P + a;
    int o[P];
#pragma unroll
    for (int k = 0; k < P; k++) o[k] = __ldg(off + k * P * P);
#pragma unroll
    for (int k = 0; k < P; k++) {
      soff[eb * P3 + (k * P + b) * P + a] = o[k];
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
        R0[B200_K12_IDX(c, a, b, qz)] = s;
      }
  }
  __syncthreads();
  // ---- y-lines, contract y with B
  if (act && a < P) {
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double in[P];
#pragma unroll
      for (int j = 0; j < P; j++) in[j] = R0[B200_K12_IDX(c, a, j, b)];
#pragma unroll
      for (int qy = 0; qy < Q; qy++) {
        double s = 0;
#pragma unroll
        for (int j = 0; j < P; j++) s += m.B[qy * P + j] * in[j];
        R1[B200_K12_IDX(c, a, qy, b)] = s;
      }
    }
  }
  __syncthreads();
  // ---- x-lines, contract x with B; d/dx in registers
  double Hx[3][Q];
  if (act) {
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double in[P], ut[Q];
#pragma unroll
      for (int i = 0; i < P; i++) in[i] = R1[B200_K12_IDX(c, i, a, b)];
#pragma unroll
      for (int qx = 0; qx < Q; qx++) {
        double s = 0;
#pragma unroll
        for (int i = 0; i < P; i++) s += m.B[qx * P + i] * in[i];
        ut[qx] = s;
        R0[B200_K12_IDX(c, qx, a, b)] = s;
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
  // ---- y-lines: d/dy -> R1;  z-lines: d/dz -> R2
  if (act) {
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double in[Q];
#pragma unroll
      for (int mm = 0; mm < Q; mm++) in[mm] = R0[B200_K12_IDX(c, a, mm, b)];
#pragma unroll
      for (int qy = 0; qy < Q; qy++) {
        double s = 0;
#pragma unroll
        for (int mm = 0; mm < Q; mm++) s += m.Gc[qy * Q + mm] * in[mm];
        R1[B200_K12_IDX(c, a, qy, b)] = s;
      }
#pragma unroll
      for (int mm = 0; mm < Q; mm++) in[mm] = R0[B200_K12_IDX(c, a, b, mm)];
#pragma unroll
      for (int qz = 0; qz < Q; qz++) {
        double s = 0;
#pragma unroll
        for (int mm = 0; mm < Q; mm++) s += m.Gc[qz * Q + mm] * in[mm];
        R2[B200_K12_IDX(c, a, b, qz)] = s;
      }
    }
  }
  __syncthreads();
  // ---- the user QFunction at the Q points of this x-line; then d/dx^T in registers
  if (act) {
    double Wx[3][Q];
#pragma unroll
    for (int qx = 0; qx < Q; qx++) {
      double H[3][3], W[3][3];
#pragma unroll
      for (int c = 0; c < 3; c++) {
        H[c][0] = Hx[c][qx];
        H[c][1] = R1[B200_K12_IDX(c, qx, a, b)];
        H[c][2] = R2[B200_K12_IDX(c, qx, a, b)];
      }
      b200_k12_point(ctx, f, grp, lane + (size_t)qx * ebt, (size_t)Q * ebt, H, W, padd);
#pragma unroll
      for (int c = 0; c < 3; c++) {
        Wx[c][qx] = W[c][0];
        R1[B200_K12_IDX(c, qx, a, b)] = W[c][1];
        R2[B200_K12_IDX(c, qx, a, b)] = W[c][2];
      }
    }
#pragma unroll
    for (int c = 0; c < 3; c++)
#pragma unroll
      for (int qx = 0; qx < Q; qx++) {
        double s = 0;
#pragma unroll
        for (int mm = 0; mm < Q; mm++) s += m.Gc[mm * Q + qx] * Wx[c][mm];
        R0[B200_K12_IDX(c, qx, a, b)] = s;
      }
  }
  __syncthreads();
  // ---- y-lines: R0 += Gc^T_y Wy
  if (act) {
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double in[Q];
#pragma unroll
      for (int mm = 0; mm < Q; mm++) in[mm] = R1[B200_K12_IDX(c, a, mm, b)];
#pragma unroll
      for (int qy = 0; qy < Q; qy++) {
        double s = R0[B200_K12_IDX(c, a, qy, b)];
#pragma unroll
        for (int mm = 0; mm < Q; mm++) s += m.Gc[mm * Q + qy] * in[mm];
        R0[B200_K12_IDX(c, a, qy, b)] = s;
      }
    }
  }
  __syncthreads();
  // ---- z-lines: v~ = R0 + Gc^T_z Wz, then B^T along z -> R1
  if (act) {
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double in[Q], vt[Q];
#pragma unroll
      for (int mm = 0; mm < Q; mm++) in[mm] = R2[B200_K12_IDX(c, a, b, mm)];
#pragma unroll
      for (int qz = 0; qz < Q; qz++) {
        double s = R0[B200_K12_IDX(c, a, b, qz)];
#pragma unroll
        for (int mm = 0; mm < Q; mm++) s += m.Gc[mm * Q + qz] * in[mm];
        vt[qz] = s;
      }
#pragma unroll
      for (int k = 0; k < P; k++) {
        double s = 0;
#pragma unroll
        for (int qz = 0; qz < Q; qz++) s += m.B[qz * P + k] * vt[qz];
        R1[B200_K12_IDX(c, a, b, k)] = s;
      }
    }
  }
  __syncthreads();
  // ---- y-lines (b = k < P): B^T along y -> R2
  if (act && b < P) {
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double in[Q];
#pragma unroll
      for (int qy = 0; qy < Q; qy++) in[qy] = R1[B200_K12_IDX(c, a, qy, b)];
#pragma unroll
      for (int j = 0; j < P; j++) {
        double s = 0;
#pragma unroll
        for (int qy = 0; qy < Q; qy++) s += m.B[qy * P + j] * in[qy];
        R2[B200_K12_IDX(c, a, j, b)] = s;
      }
    }
  }
  __syncthreads();
  // ---- x-lines (a = j < P, b = k < P): B^T along x -> nodal output, interlaced [node][component] in R0/R1
  if (act && a < P && b < P) {
    double *Rn = R0 + ((b * P + a) * P) * 3;
#pragma unroll
    for (int c = 0; c < 3; c++) {
      double in[Q];
#pragma unroll
      for (int qx = 0; qx < Q; qx++) in[qx] = R2[B200_K12_IDX(c, qx, a, b)];
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
  // ---- scatter in L-vector order: flat sweep over (element, node, component), component fastest
  {
    constexpr int NIT = (EB * 3 * P3 + NT - 1) / NT;
    const int total = ebn * 3 * P3;
    double *ev = evec ? evec + (size_t)blk * EB * 3 * P3 : nullptr;
#pragma unroll
    for (int it = 0; it < NIT; it++) {
      const int fi = tid + it * NT;
      if (fi < total) {
        const int el = fi / (3 * P3), r = fi - el * (3 * P3), node = r / 3;
        const double v = smem[el * SE + r];
        if (ev) ev[fi] = v;
        else atomicAdd(y + soff[el * P3 + node] + (r - node * 3), v);
      }
    }
  }
}

#undef B200_K12_IDX
#endif
