"""Coarse-level assembly on the device (CeedOperatorLinearAssemble[Symbolic], stencil Galerkin product) against
the oracle: the assembled matrix must be the matrix of the oracle's Jacobian operator (column by column), and
the solver must take the same iterations whichever way the matrix was built.  FP64, 1e-12 relative."""
import numpy as np
import pytest
import torch

from helpers import OracleProblem, dense_from_stencil, lattice_ids, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-12


@pytest.fixture(scope="module")
def G():
    import gpu_helpers
    return gpu_helpers


def _coo_dense(g, level):
    op = g.data[level].opJacob
    rows, cols = op.linear_assemble_symbolic()
    vals = g.ceed.Vector(rows.size)
    op.linear_assemble(vals)
    v = vals.to_numpy()
    vals.destroy()
    n = 3 * g.mesh.num_nodes(g.degrees[level])
    A = np.zeros((n, n))
    np.add.at(A, (rows, cols), v)
    return A, rows, cols


@pytest.mark.parametrize("problem,n,p,qextra", [("linElas", 2, 1, 0), ("hyperSS", (3, 2, 2), 2, 0), ("hyperFS", (2, 3, 2), 2, 0),
                                                ("hyperFS", (5, 2, 3), 4, 0), ("hyperFS", 2, 3, 1), ("hyperSS", (17, 1, 1), 1, 1)])
def test_linear_assemble_is_the_oracle_jacobian(G, problem, n, p, qextra):
    g = G.GpuProblem(problem, n, p, qextra=qextra)
    assert g.degrees[0] == 1
    g.residual()  # the state (gradu) the Jacobian is linearised about
    A, rows, cols = _coo_dense(g, 0)
    o = OracleProblem(problem, n, p, pl=1, qextra=qextra)
    assert rows.size == 576 * o.nelem
    # symbolic pattern: 24 x 24 block per element over the element's dofs
    off = o.offsets.reshape(-1, 8)
    eldofs = (off[:, :, None] + np.arange(3)[None, None, :]).reshape(-1, 24)
    np.testing.assert_array_equal(rows.reshape(-1, 24, 24), np.broadcast_to(eldofs[:, None, :], (o.nelem, 24, 24)))
    np.testing.assert_array_equal(cols.reshape(-1, 24, 24), np.broadcast_to(eldofs[:, :, None], (o.nelem, 24, 24)))
    Ao = np.stack([o.jacobian(e) for e in np.eye(o.lsize)], axis=1)
    assert rel_err(A, Ao) < TOL
    assert rel_err(A, A.T) < TOL                      # hyperelastic tangent: symmetric
    assert rel_err(np.diag(A), o.diagonal()) < TOL    # consistent with LinearAssembleDiagonal
    assert rel_err(np.diag(A), g.diagonal(0)) < TOL


def test_linear_assemble_refuses_other_levels(G):
    g = G.GpuProblem("hyperFS", 2, 2)
    from ceedpetscsolid_b200.ceed import CeedError
    with pytest.raises(CeedError, match="trilinear"):
        g.data[1].opJacob.linear_assemble_symbolic()
    v = g.ceed.Vector(10)
    with pytest.raises(CeedError, match="entries"):
        g.data[0].opJacob.linear_assemble(v)


@pytest.mark.parametrize("Nc", [(2, 2, 2), (3, 2, 4), (5, 5, 3)])
def test_stencil_galerkin_kernel_is_PtAP(Nc):
    """A_H from the kernel == dense P^T A P with the trilinear lattice prolongation"""
    from ceedpetscsolid_b200.ceed import lib, b2
    from ceedpetscsolid_b200.solver import _lattice_prolong_cpu
    Nf = tuple(2 * v - 1 for v in Nc)
    nf, nc = 3 * int(np.prod(Nf)), 3 * int(np.prod(Nc))
    rng = np.random.default_rng(3)
    sv = rng.standard_normal((81, nf))
    # entries that point outside the fine lattice are zero by construction of the assembled matrix
    i, j, k = lattice_ids(Nf)
    for o in range(27):
        dx, dy, dz = o % 3 - 1, (o // 3) % 3 - 1, o // 9 - 1
        bad = ~((i + dx >= 0) & (i + dx < Nf[0]) & (j + dy >= 0) & (j + dy < Nf[1]) & (k + dz >= 0) & (k + dz < Nf[2]))
        sv[o * 3:(o + 1) * 3, np.repeat(bad, 3)] = 0
    Af = dense_from_stencil(sv, Nf)
    Pm = np.stack([_lattice_prolong_cpu(Nc, torch.from_numpy(e)).numpy().reshape(-1) for e in np.eye(nc)], axis=1)
    AH = Pm.T @ Af @ Pm
    d_f = torch.from_numpy(sv).cuda()
    d_c = torch.full((81, nc), np.nan, dtype=torch.float64, device="cuda")
    b2(lib.b200_stencil27_galerkin(Nc[0], Nc[1], Nc[2], d_f.data_ptr(), d_c.data_ptr()))
    torch.cuda.synchronize()
    got = d_c.cpu().numpy()
    assert np.isfinite(got).all()
    assert rel_err(dense_from_stencil(got, Nc), AH) < 1e-13
    # and nothing is stored for neighbours outside the coarse lattice
    i, j, k = lattice_ids(Nc)
    for o in range(27):
        dx, dy, dz = o % 3 - 1, (o // 3) % 3 - 1, o // 9 - 1
        bad = ~((i + dx >= 0) & (i + dx < Nc[0]) & (j + dy >= 0) & (j + dy < Nc[1]) & (k + dz >= 0) & (k + dz < Nc[2]))
        assert not got[o * 3:(o + 1) * 3, np.repeat(bad, 3)].any()


def test_solver_iterations_do_not_depend_on_how_the_coarse_matrix_is_built():
    from ceedpetscsolid_b200.elasticity import AppCtx, Elasticity
    outs = []
    for assemble in ("color", "coo"):
        app = AppCtx(problem="hyperFS", degree=2, n=(8, 4, 4), num_steps=2, perturb=0.05)
        el = Elasticity(app, assemble=assemble)
        assert (el.pc.coarse.coo is not None) == (assemble == "coo")
        out = el.solve()
        outs.append((out["snes_its"], out["ksp_its"], out["coarse_its"], el.pc.coarse.svals.clone(), el.U.clone()))
    assert outs[0][:3] == outs[1][:3]
    assert rel_err(outs[1][3].cpu().numpy(), outs[0][3].cpu().numpy()) < TOL
    assert rel_err(outs[1][4].cpu().numpy(), outs[0][4].cpu().numpy()) < 1e-9
