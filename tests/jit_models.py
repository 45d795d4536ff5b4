"""User QFunction sources for the tests of the kernels around JIT-compiled QFunctions (K12, K13, K14)."""

# A linear-elastic model with extra passive fields, its active fields away from index 0 (fields map by declaration
# order): in = [scale (1), du (9, gradient), qdata (10)], out = [sdiag (3), dv (9, gradient), energy (1)].
# stress = s (lambda tr(eps) I + 2 mu eps) with s = 1 + scale / 2; sdiag = the stress diagonal, energy = stress:eps/2.
EXTRA_FIELDS = r"""#include <ceed.h>
typedef struct { CeedScalar nu, E; } ExtraPhysics;

CEED_QFUNCTION(ExtraF)(void *ctx, const CeedInt Q, const CeedScalar *const *in, CeedScalar *const *out) {
  const CeedScalar *scale = in[0];
  const CeedScalar(*du)[3][CEED_Q_VLA] = (const CeedScalar(*)[3][CEED_Q_VLA])in[1];
  const CeedScalar(*qd)[CEED_Q_VLA] = (const CeedScalar(*)[CEED_Q_VLA])in[2];
  CeedScalar(*sdiag)[CEED_Q_VLA] = (CeedScalar(*)[CEED_Q_VLA])out[0];
  CeedScalar(*dv)[3][CEED_Q_VLA] = (CeedScalar(*)[3][CEED_Q_VLA])out[1];
  CeedScalar *energy = out[2];
  const ExtraPhysics *p = (const ExtraPhysics *)ctx;
  const CeedScalar mu = p->E / (2 * (1 + p->nu)), lambda = p->E * p->nu / ((1 + p->nu) * (1 - 2 * p->nu));
  CeedPragmaSIMD
  for (CeedInt i = 0; i < Q; i++) {
    CeedScalar X[3][3], H[3][3], eps[3][3], sig[3][3];
    const CeedScalar wdetJ = qd[0][i], s = 1 + 0.5 * scale[i];
    for (int a = 0; a < 3; a++)
      for (int b = 0; b < 3; b++) X[a][b] = qd[1 + 3 * a + b][i];
    for (int c = 0; c < 3; c++)
      for (int k = 0; k < 3; k++) {
        CeedScalar t = 0;
        for (int m = 0; m < 3; m++) t += X[m][k] * du[m][c][i];
        H[c][k] = t;
      }
    for (int a = 0; a < 3; a++)
      for (int b = 0; b < 3; b++) eps[a][b] = (H[a][b] + H[b][a]) / 2;
    const CeedScalar tr = eps[0][0] + eps[1][1] + eps[2][2];
    CeedScalar e = 0;
    for (int a = 0; a < 3; a++)
      for (int b = 0; b < 3; b++) {
        sig[a][b] = s * ((a == b ? lambda * tr : 0) + 2 * mu * eps[a][b]);
        e += sig[a][b] * eps[a][b];
      }
    for (int a = 0; a < 3; a++) sdiag[a][i] = sig[a][a];
    energy[i] = 0.5 * e * wdetJ;
    for (int k = 0; k < 3; k++)
      for (int c = 0; c < 3; c++) {
        CeedScalar t = 0;
        for (int m = 0; m < 3; m++) t += X[k][m] * sig[c][m];
        dv[k][c][i] = t * wdetJ;
      }
  }
  return 0;
}
"""
EXTRA_IN, EXTRA_OUT = [1, 9, 10], [3, 9, 1]


# The field-count and width limits of K11 / K12: B200_JIT_MAXF = 8 fields each way, passive widths 1 to
# B200_JIT_MAX_FIELD = 64.  The active gradient g is the LAST input (7) and a MIDDLE output (3).  The context is 256
# doubles k (B200_JIT_MAX_CTX = 2048 bytes); k[255], its last 8 bytes, enters every output.  With x the passive input
# components numbered through the fields in order (92 of them), passive output component m (numbered the same way,
# 93 of them) is
#     k[m] x[7m mod 92] + x[(13m + 5) mod 92] (1 + g[m mod 9] / 4) + (m + 1) k[255]
# (7m mod 92 reaches every x), and active output component j is
#     sum_d k[100 + 9j + d] g[d] + x[(11j + 3) mod 92] g[(j + 4) mod 9] + k[255] x[40 + j],
# so a swapped field, component, point or element changes the answer.  Fields are [comp][Q], indexed with Q itself:
# the same text runs with Q = 1 on the device and Q = nq on the host.
EDGE_FIELDS = r"""#include <ceed.h>

CEED_QFUNCTION(EdgeF)(void *ctx, const CeedInt Q, const CeedScalar *const *in, CeedScalar *const *out) {
  const CeedScalar *k = (const CeedScalar *)ctx;
  const int win[7] = {1, 2, 7, 64, 3, 5, 10}, wout[8] = {2, 64, 1, 9, 7, 3, 5, 11};
  for (CeedInt i = 0; i < Q; i++) {
    CeedScalar x[92], g[9];
    int n = 0;
    for (int f = 0; f < 7; f++)
      for (int c = 0; c < win[f]; c++) x[n++] = in[f][c * Q + i];
    for (int d = 0; d < 9; d++) g[d] = in[7][d * Q + i];
    int m = 0;
    for (int f = 0; f < 8; f++) {
      if (f == 3) {
        for (int j = 0; j < 9; j++) {
          CeedScalar s = x[(11 * j + 3) % 92] * g[(j + 4) % 9] + k[255] * x[40 + j];
          for (int d = 0; d < 9; d++) s += k[100 + 9 * j + d] * g[d];
          out[3][j * Q + i] = s;
        }
        continue;
      }
      for (int c = 0; c < wout[f]; c++, m++)
        out[f][c * Q + i] = k[m] * x[(7 * m) % 92] + x[(13 * m + 5) % 92] * (1 + 0.25 * g[m % 9]) + (m + 1) * k[255];
    }
  }
  return 0;
}
"""
EDGE_IN, EDGE_OUT, EDGE_AI, EDGE_AO, EDGE_CTX = [1, 2, 7, 64, 3, 5, 10, 9], [2, 64, 1, 9, 7, 3, 5, 11], 7, 3, 256


# A non-symmetric linear model: dv = wdetJ dXdx sigma, sigma_i = sum_j K[9 i + j] H_j, H = the physical gradient of du,
# i = c*3 + k; K (the context, 81 doubles) is not symmetric, so neither is the point tangent.
# in = [du (9, gradient), qdata (10)], out = [dv (9, gradient)].
NONSYM = r"""#include <ceed.h>
CEED_QFUNCTION(NonSymdF)(void *ctx, const CeedInt Q, const CeedScalar *const *in, CeedScalar *const *out) {
  const CeedScalar *K = (const CeedScalar *)ctx;
  const CeedScalar(*du)[3][CEED_Q_VLA] = (const CeedScalar(*)[3][CEED_Q_VLA])in[0];
  const CeedScalar(*qd)[CEED_Q_VLA] = (const CeedScalar(*)[CEED_Q_VLA])in[1];
  CeedScalar(*dv)[3][CEED_Q_VLA] = (CeedScalar(*)[3][CEED_Q_VLA])out[0];
  for (CeedInt i = 0; i < Q; i++) {
    CeedScalar X[3][3], H[9], sig[9];
    for (int a = 0; a < 3; a++)
      for (int b = 0; b < 3; b++) X[a][b] = qd[1 + 3 * a + b][i];
    for (int c = 0; c < 3; c++)
      for (int k = 0; k < 3; k++) {
        CeedScalar t = 0;
        for (int m = 0; m < 3; m++) t += X[m][k] * du[m][c][i];
        H[c * 3 + k] = t;
      }
    for (int r = 0; r < 9; r++) {
      CeedScalar t = 0;
      for (int s = 0; s < 9; s++) t += K[9 * r + s] * H[s];
      sig[r] = t;
    }
    for (int k = 0; k < 3; k++)
      for (int c = 0; c < 3; c++) {
        CeedScalar t = 0;
        for (int m = 0; m < 3; m++) t += X[k][m] * sig[c * 3 + m];
        dv[k][c][i] = t * qd[0][i];
      }
  }
  return 0;
}
"""
NONSYM_IN, NONSYM_OUT, NONSYM_CTX = [9, 10], [9], 81
