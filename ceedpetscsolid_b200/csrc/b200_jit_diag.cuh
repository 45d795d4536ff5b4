// K14: the operator diagonal around a user QFunction compiled at run time ("/gpu/b200:jit").
//
// Device-only template.  It is not compiled into the library: the build embeds it as a string (b200_jit.cu), and NVRTC
// compiles it together with the user's program and a generated prefix that defines, before this text:
//   B200_K14_P, B200_K14_Q                       the basis (P, Q), one of B200_FOR_PQ
//   B200_K14_SY, _SZ, _SC, _SE, _EB, _NT         the shared-memory lattice of b200_apply_smem_layout(P, Q) (K12's)
//   b200_jit_ctx_t, b200_k14_fields_t            the context bytes and the input field pointers (by field index)
//   b200_k14_prefetch(f, grp, npts)              one bulk L2 prefetch per passive input slab of the group
//   b200_k14_point(ctx, f, grp, pos, cs, c, fold)
//       the tangent of component c at one point: for m = 0, 1, 2 the passive inputs loaded from their q-blocked slabs
//       (field i at f.in[i] + grp * size_i + pos + comp * cs; L1 hits after m = 0, and no registers held across the
//       calls), the user function called with Q = 1 and the active input set to the unit vector e_(m,c)
//       (in[m*3 + c] = 1), and fold(m, v) with v[k] = out_active[k*3 + c].  Passive outputs are discarded; the return
//       code is ignored.
// and, after it, the two extern "C" kernels that call b200_k14_body<true> (full groups) and <false> (the tail group).
//
// With in[m*3 + b] = H[b][m], out[k*3 + a] = W[a][k] and D[a k][b m] = dW[a][k] / dH[b][m] (the K12 convention),
// v[k] = D[c k][c m] and the diagonal entry of node n, component c is
//   diag_e[n][c] = sum_q sum_{k,m} G_k(q,n) D_q[c k][c m] G_m(q,n),
// G the tensor shape gradients.  Since G_k G_m = G_m G_k, only the six terms of k_fused_diag (b200_fused.cu) appear,
//   A_dd = D[c d][c d],   A_dd' = D[c d][c d'] + D[c d'][c d]  (d < d'),
// which holds whether or not the user tangent is symmetric.  This is the diagonal of the operator only if the user
// function is linear in its active input, as every Jacobian QFunction is (libCEED assumes the same).
//
// The contraction is K3's: one sweep per component c; in each, the x-line owner forms the six A_t at its Q points,
// parks them in its own line of the lattices and contracts them along x with B.B, B.D or D.D, then the y and z stages
// merge the terms by their selectors through nine single-component lattices per element.  Output: FP64 atomics at offsets + c, or plain stores to an
// E-vector [e][node][comp] that the caller sums in a fixed order.
#ifndef B200_JIT_DIAG_CUH
#define B200_JIT_DIAG_CUH

struct b200_k14_mats_t {
  double M[3][B200_K14_Q * B200_K14_P];  // [0] B.B  [1] B.D  [2] D.D  (element-wise, [Q][P])
};

#define B200_K14_IDX(c, x, y, z) ((c) * SC + (z) * SZ + (y) * SY + (x))

template <bool FULL>
__device__ __forceinline__ void b200_k14_body(const b200_k14_mats_t &dm, const b200_jit_ctx_t &ctx,
                                              const b200_k14_fields_t &f, const int nelem,
                                              const int *__restrict__ offsets, double *__restrict__ diag,
                                              double *__restrict__ evec) {
  constexpr int P = B200_K14_P, Q = B200_K14_Q, T = Q * Q, P3 = P * P * P;
  constexpr int SY = B200_K14_SY, SZ = B200_K14_SZ, SC = B200_K14_SC, SE = B200_K14_SE, EB = B200_K14_EB;
  static_assert(9 * SC <= SE, "nine single-component lattices per element");
  static_assert(T * EB <= B200_K14_NT, "one thread per x-line");
  // selectors of term t = (d, d') per axis: (d == axis) + (d' == axis); Voigt order 00, 11, 22, 12, 02, 01
  constexpr int SELX[6] = {2, 0, 0, 0, 1, 1}, SELY[6] = {0, 2, 0, 1, 0, 1}, SELZ[6] = {0, 0, 2, 1, 1, 0};
  extern __shared__ double smem[];
  const int tid = threadIdx.x;
  const int t = tid / EB, eb = tid - t * EB, a = t % Q, b = t / Q;
  const int blk = blockIdx.x;
  const int rem = nelem - blk * EB;
  const int ebn = FULL ? EB : (rem < EB ? rem : EB);
  const bool act = t < T && (FULL || eb < ebn);
  const int e = blk * EB + eb;
  double *R = smem + eb * SE;  // 9 single-component lattices: terms 0..5, then the three z-selector sums
  // q-blocked slabs of the passive inputs: group base (per component), this lane, the plane stride
  const size_t grp = (size_t)blk * EB * Q * T;
  const size_t ebt = FULL ? (size_t)(EB * T) : (size_t)ebn * T;
  const size_t lane = FULL ? (size_t)tid : (size_t)(t * ebn + eb);
  // the group's slabs in one bulk L2 request each: the three sweeps then read them from L2
  if (tid == 0) b200_k14_prefetch(f, grp, Q * ebt);

#pragma unroll 1
  for (int c = 0; c < 3; c++) {
    if (act) {
      // A_t at the line's Q points, parked in the thread's own line of lattices 0..5 (no barrier): only the user
      // function's state is live across its calls
#pragma unroll 1
      for (int qx = 0; qx < Q; qx++) {
        // call m gives column m of the block, v[k] = D[c k][c m]: fold it into the terms at once (t = 3, 4, 5 are the
        // pairs 12, 02, 01, each the sum of its two entries)
        double A[6] = {0, 0, 0, 0, 0, 0};
        b200_k14_point(ctx, f, grp, lane + (size_t)qx * ebt, (size_t)Q * ebt, c, [&](const int m, const double *v) {
          if (m == 0) { A[0] = v[0]; A[4] += v[2]; A[5] += v[1]; }
          if (m == 1) { A[1] = v[1]; A[3] += v[2]; A[5] += v[0]; }
          if (m == 2) { A[2] = v[2]; A[3] += v[1]; A[4] += v[0]; }
        });
#pragma unroll
        for (int tt = 0; tt < 6; tt++) R[B200_K14_IDX(tt, qx, a, b)] = A[tt];
      }
      // x-stage: S_t[i] = sum_qx A_t(qx) Mx[sel_x(t)][qx][i], written over the same line
#pragma unroll
      for (int tt = 0; tt < 6; tt++) {
        double in[Q];
#pragma unroll
        for (int qx = 0; qx < Q; qx++) in[qx] = R[B200_K14_IDX(tt, qx, a, b)];
#pragma unroll
        for (int i = 0; i < P; i++) {
          double s = 0;
#pragma unroll
          for (int qx = 0; qx < Q; qx++) s += dm.M[SELX[tt]][qx * P + i] * in[qx];
          R[B200_K14_IDX(tt, i, a, b)] = s;
        }
      }
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
        for (int qy = 0; qy < Q; qy++) in[qy] = R[B200_K14_IDX(tt, a, qy, b)];
#pragma unroll
        for (int j = 0; j < P; j++)
#pragma unroll
          for (int qy = 0; qy < Q; qy++) Y[SELZ[tt]][j] += dm.M[SELY[tt]][qy * P + j] * in[qy];
      }
#pragma unroll
      for (int s = 0; s < 3; s++)
#pragma unroll
        for (int j = 0; j < P; j++) R[B200_K14_IDX(6 + s, a, j, b)] = Y[s][j];
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
        for (int qz = 0; qz < Q; qz++) in[qz] = R[B200_K14_IDX(6 + s, a, b, qz)];
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
        for (int k = 0; k < P; k++) atomicAdd(diag + __ldg(offsets + (size_t)e * P3 + (k * P + b) * P + a) + c, acc[k]);
      }
    }
    // the next component's x-stage writes lattices 0..5 (their readers passed the second barrier) and its y-stage
    // writes 6..8 only behind the next barrier, which no thread reaches before finishing this z-stage
  }
}

#undef B200_K14_IDX
#endif
