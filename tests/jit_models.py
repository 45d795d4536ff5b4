"""User QFunction sources for the tests of the fused kernel around JIT-compiled QFunctions (K12)."""

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
