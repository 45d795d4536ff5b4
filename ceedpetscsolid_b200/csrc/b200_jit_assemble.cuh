// K13: element matrices of a trilinear (P = 2) level around a user QFunction compiled at run time ("/gpu/b200:jit"),
// in the CeedOperatorLinearAssemble layout of k_assemble_p1 (b200_assemble.cu): values[(e*24 + col)*24 + row],
// element dof = node*3 + component, node = ix + 2 iy + 4 iz.
//
// Device-only template.  It is not compiled into the library: the build embeds it as a string (b200_jit.cu), and NVRTC
// compiles it together with the user's program and a generated prefix that defines, before this text:
//   B200_K13_Q                     the number of 1D quadrature points (P = 2)
//   B200_K13_EB, B200_K13_NT       elements per CTA (the q-blocked group, b200_elems_per_block(Q)) and threads = 24 EB
//   B200_K13_CH                    points whose tangent a CTA holds in shared memory at once (CH <= NT)
//   b200_jit_ctx_t, b200_k13_fields_t            the context bytes and the input field pointers (by field index)
//   b200_k13_point(ctx, f, grp, pos, cs, d)
//       the point tangent at one point: the passive inputs loaded once from their q-blocked slabs (field i at
//       f.in[i] + grp * size_i + pos + comp * cs), then the user function called 9 times with Q = 1 and the active
//       input set to the unit vectors, d[s*9 + o] = out_active[o] for in_active = e_s.  Passive outputs are discarded.
// and, after it, the two extern "C" kernels that call b200_k13_body<true> (full groups) and <false> (the tail group).
//
// With in[s = m*3 + b] = H[b][m] and out[o = k*3 + a] = W[a][k] (the K12 convention), d[(m*3 + b)*9 + k*3 + a] is
// dW[a][k] / dH[b][m].  The element matrix is then
//   K_e[(i,a)][(j,b)] = sum_q sum_{k,m} G_{i,k}(q) D_q[a k][b m] G_{j,m}(q)
// with G the trilinear reference shape gradients.  This equals the Jacobian only if the user function is linear in its
// active input, as every Jacobian QFunction is (libCEED's CeedOperatorLinearAssembleQFunction assumes the same).
//
// The positions of a group are walked in q-blocked order p = qx*(ebn*Q^2) + t*ebn + e (t = qy + Q*qz), CH at a time:
// thread p of a chunk writes the tangent of position p to shared memory (coalesced passive loads), then every thread
// (element e, column col) adds the chunk's points of its element to its 24 row sums in registers.  Each entry is a
// sum in a fixed order: no atomics, results are bit-identical from run to run.
#ifndef B200_JIT_ASSEMBLE_CUH
#define B200_JIT_ASSEMBLE_CUH

struct b200_k13_mats_t {
  double B[B200_K13_Q * 2];  // interp1d [Q][2]
  double D[B200_K13_Q * 2];  // grad1d   [Q][2]
};

template <bool FULL>
__device__ __forceinline__ void b200_k13_body(const b200_k13_mats_t &m, const b200_jit_ctx_t &ctx,
                                              const b200_k13_fields_t &f, const int nelem,
                                              double *__restrict__ values) {
  constexpr int Q = B200_K13_Q, T = Q * Q, Q3 = Q * Q * Q, EB = B200_K13_EB, CH = B200_K13_CH;
  static_assert(B200_K13_NT == 24 * EB && CH <= B200_K13_NT, "one thread per (element, column); CH <= threads");
  extern __shared__ double sd[];  // [CH][81] point tangents
  const int tid = threadIdx.x;
  const int col = tid / EB, eb = tid - col * EB;
  const int blk = blockIdx.x;
  const int rem = nelem - blk * EB;
  const int ebn = FULL ? EB : (rem < EB ? rem : EB);
  const int npos = ebn * Q3;
  const bool act = eb < ebn;
  // q-blocked slabs of the passive inputs: group base (per component), the component stride
  const size_t grp = (size_t)blk * EB * Q3, cs = (size_t)npos;
  const int j = col / 3, cb = col - 3 * j;
  const bool jx = j & 1, jy = (j >> 1) & 1, jz = j >> 2;
  double acc[24];
#pragma unroll
  for (int r = 0; r < 24; r++) acc[r] = 0;
#pragma unroll 1
  for (int c0 = 0; c0 < npos; c0 += CH) {
    if (tid < CH && c0 + tid < npos) b200_k13_point(ctx, f, grp, (size_t)(c0 + tid), cs, sd + tid * 81);
    __syncthreads();
    if (act) {
      const int cend = c0 + CH < npos ? c0 + CH : npos;
#pragma unroll 1
      for (int p = c0 + (eb - c0 % ebn + ebn) % ebn; p < cend; p += ebn) {
        const int pi = p / ebn, qx = pi / T, t = pi - qx * T, qz = t / Q, qy = t - qz * Q;
        const double *d = sd + (p - c0) * 81;
        const double bx[2] = {m.B[qx * 2], m.B[qx * 2 + 1]}, dx[2] = {m.D[qx * 2], m.D[qx * 2 + 1]};
        const double by[2] = {m.B[qy * 2], m.B[qy * 2 + 1]}, dy[2] = {m.D[qy * 2], m.D[qy * 2 + 1]};
        const double bz[2] = {m.B[qz * 2], m.B[qz * 2 + 1]}, dz[2] = {m.D[qz * 2], m.D[qz * 2 + 1]};
        // column gradient: node j, component cb (selects, not run-time indices: the pairs stay in registers)
        const double cbx = jx ? bx[1] : bx[0], cdx = jx ? dx[1] : dx[0], cby = jy ? by[1] : by[0];
        const double cdy = jy ? dy[1] : dy[0], cbz = jz ? bz[1] : bz[0], cdz = jz ? dz[1] : dz[0];
        const double g[3] = {cdx * cby * cbz, cbx * cdy * cbz, cbx * cby * cdz};
        double W[3][3];
#pragma unroll
        for (int a = 0; a < 3; a++)
#pragma unroll
          for (int k = 0; k < 3; k++) {
            double s = 0;
#pragma unroll
            for (int mm = 0; mm < 3; mm++) s += d[(mm * 3 + cb) * 9 + k * 3 + a] * g[mm];
            W[a][k] = s;
          }
#pragma unroll
        for (int i = 0; i < 8; i++) {
          const int ix = i & 1, iy = (i >> 1) & 1, iz = i >> 2;
          const double g0 = dx[ix] * by[iy] * bz[iz], g1 = bx[ix] * dy[iy] * bz[iz], g2 = bx[ix] * by[iy] * dz[iz];
#pragma unroll
          for (int a = 0; a < 3; a++) acc[i * 3 + a] += g0 * W[a][0] + g1 * W[a][1] + g2 * W[a][2];
        }
      }
    }
    __syncthreads();
  }
  if (act) {
    double *out = values + ((size_t)(blk * EB + eb) * 24 + col) * 24;
#pragma unroll
    for (int r = 0; r < 24; r += 2) *reinterpret_cast<double2 *>(out + r) = make_double2(acc[r], acc[r + 1]);
  }
}

#endif
