"""Shared set-up of the AMG tests: element matrices of the p = 1 operator from the oracle, and the Newton-Krylov-p-MG
solve of oracle_levels with the smoothed-aggregation AMG coarse solve."""
import numpy as np
import torch

from ceedpetscsolid_b200 import matops, solver
from ceedpetscsolid_b200.amg import MAX_COARSE_DOFS, SmoothedAggregationAMG
from helpers import PHYS
from oracle import oracle
from oracle_levels import OracleLevel, OracleShared, OracleTransfer


def oracle_element_matrices(mesh, problem="linElas"):
    """(E, 24, 24) element matrices of the trilinear Jacobian (linearised at zero displacement), element dof =
    node*3 + component: 24 applies of the oracle operator on a discontinuous copy of the mesh."""
    E = mesh.nelem
    B, D, _, _ = oracle.basis_1d(2, 2, 0)
    qdata = oracle.setup_geo(E, 2, mesh.offsets(1), mesh.coord_lvector())
    gradu = np.zeros((E, 9, 8)) if oracle.PROBLEMS[problem][2] else None
    off = (np.arange(E * 8, dtype=np.int32) * 3).reshape(E, 8)
    K = np.zeros((E, 24, 24))
    for col in range(24):
        x = np.zeros((E, 24))
        x[:, col] = 1.0
        y = oracle.operator_apply(problem, True, PHYS, E, 2, 2, B, D, off, qdata, gradu, x.reshape(-1))
        K[:, :, col] = y.reshape(E, 24)
    return K


class Coo:
    """CPU stand-in of GpuLevel.enable_coo: element matrices in CeedOperatorLinearAssemble layout [e][col][row]."""

    def __init__(self, mesh, K):
        self.elem_nodes = torch.from_numpy(mesh.offsets(1).reshape(-1, 8).astype(np.int64) // 3)
        self._v = torch.from_numpy(np.ascontiguousarray(K.transpose(0, 2, 1)).reshape(-1))

    def values(self):
        return self._v


class CoarseStub:
    """What SmoothedAggregationAMG.setup reads from PMultigrid's p = 1 matrix object."""

    def __init__(self, coo):
        self.coo = coo


def assembled(mesh, K, dm):
    """scipy CSR of the p = 1 matrix with constrained rows/columns masked (unit diagonal)"""
    import scipy.sparse as sp
    E = mesh.nelem
    eld = (mesh.offsets(1).reshape(E, 8)[:, :, None] + np.arange(3)).reshape(E, 24)
    rows = np.repeat(eld, 24, axis=1).reshape(-1)
    cols = np.tile(eld, (1, 24)).reshape(-1)
    A = sp.csr_matrix((K.reshape(-1), (rows, cols)), shape=(dm.lsize, dm.lsize))
    free = np.repeat(~dm.bc_nodes, 3).astype(float)
    A = sp.diags(free) @ A @ sp.diags(free) + sp.diags(1.0 - free)
    return A.tocsr()


def amg_oracle_solve(app, max_coarse=MAX_COARSE_DOFS, log=None, **kw):
    """oracle_levels.oracle_solve with coarse='amg' (unstructured or box meshes, one rank, masked layout).
    Returns (summary, U, preconditioner)."""
    sh = OracleShared(app, masked=True)
    L = len(sh.degrees)
    levels = [OracleLevel(sh, l, l == L - 1) for l in range(L)]
    transfers = [None] + [OracleTransfer(sh, levels[l - 1], levels[l]) for l in range(1, L)]
    V = solver.Vec()
    V.consistent = {lev.dm.nglobal: lev.dm.make_consistent for lev in levels}
    amg = SmoothedAggregationAMG(levels[0].dm, sh.mesh, max_coarse=max_coarse)
    pc = solver.PMultigrid(V, levels, transfers, amg=amg)
    U = levels[-1].dm.create_global_vector(matops.MEM_HOST)
    out = solver.newton_solve(V, levels[-1], pc, U, num_increments=app.num_steps, log=log, **kw)
    return out, U, pc
