"""`/gpu/b200:deterministic`: the transposed restriction of every operator (residual, Jacobian, diagonal,
transfers, generic path) writes an E-vector and sums it per L-vector entry in ascending (element, node) order --
the order of the serial /cpu/self scatter behind CeedOperatorApply (/root/reference/src/matops.c:46) -- instead
of FP64 atomics.  Results: bit-identical from run to run, within 1e-12 of the oracle."""
import numpy as np
import pytest

from helpers import OracleProblem, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-12


DET = "/gpu/b200:deterministic"


@pytest.mark.parametrize("problem,n,p,perm", [("hyperFS", (5, 3, 3), 4, None), ("hyperSS", 4, 3, 7), ("linElas", 5, 2, None)])
def test_deterministic_mode_matches_oracle_and_is_bitwise_reproducible(problem, n, p, perm):
    import gpu_helpers as G
    from oracle import oracle
    g = G.GpuProblem(problem, n, p, node_perm_seed=perm, resource=DET)
    assert g.ceed.is_deterministic and "deterministic" in g.ceed.resource
    o = OracleProblem(problem, n, p, node_perm_seed=perm)
    y0 = g.residual()
    assert g.fine.opApply.is_fused
    assert rel_err(y0, o.to_perm(o.residual_fine(o.u_fine))) < TOL
    assert np.array_equal(y0, g.residual())
    rng = np.random.default_rng(3)
    fine = len(g.degrees) - 1
    for level, deg in enumerate(g.degrees):
        ol = OracleProblem(problem, n, p, pl=deg, node_perm_seed=perm if level == fine else None)
        x = rng.standard_normal(ol.lsize)
        y1 = g.jacobian(level, x)
        assert rel_err(y1, ol.jacobian(x)) < TOL
        assert np.array_equal(y1, g.jacobian(level, x)), "Jacobian apply differs between two runs"
        d1 = g.diagonal(level)
        assert rel_err(d1, ol.diagonal()) < TOL
        assert np.array_equal(d1, g.diagonal(level))
    if perm is None:
        for level in range(1, len(g.degrees)):
            pc, pf = g.degrees[level - 1], g.degrees[level]
            offc, offf = g.mesh.offsets(pc), g.mesh.offsets(pf)
            lc, lf = g.mesh.lsize(pc), g.mesh.lsize(pf)
            c, f = rng.standard_normal(lc), rng.standard_normal(lf)
            d = g.data[level]
            yp = g.apply(d.opProlong, c, lf)
            yr = g.apply(d.opRestrict, f, lc)
            assert rel_err(yp, oracle.transfer(False, g.mesh.nelem, pc + 1, pf + 1, offc, offf, c, lf)) < TOL
            assert rel_err(yr, oracle.transfer(True, g.mesh.nelem, pc + 1, pf + 1, offc, offf, f, lc)) < TOL
            assert np.array_equal(yp, g.apply(d.opProlong, c, lf)) and np.array_equal(yr, g.apply(d.opRestrict, f, lc))


def test_deterministic_generic_path_and_range_apply_is_refused():
    import gpu_helpers as G
    from ceedpetscsolid_b200 import ceed as libceed
    g = G.GpuProblem("hyperFS", 2, 3, qextra=2, multigrid="none", resource=DET)    # (P,Q) = (4,6): generic kernels
    o = OracleProblem("hyperFS", 2, 3, qextra=2)
    assert not g.fine.opApply.is_fused
    y = g.residual()
    assert rel_err(y, o.residual_fine(o.u_fine)) < TOL and np.array_equal(y, g.residual())
    x = np.random.default_rng(3).standard_normal(o.lsize)
    assert rel_err(g.jacobian(0, x), o.jacobian(x)) < TOL
    g2 = G.GpuProblem("hyperFS", 4, 2, resource=DET)
    n = g2.mesh.lsize(2)
    xc, yc = g2.ceed.Vector(n), g2.ceed.Vector(n)
    xc.set_value(1.0); yc.set_value(0.0)
    with pytest.raises(libceed.CeedError, match="deterministic"):
        g2.data[-1].opJacob.apply_add_range(xc, yc, 0, 16)


def test_atomic_and_deterministic_modes_agree_to_roundoff():
    import gpu_helpers as G
    ga = G.GpuProblem("hyperFS", 4, 4)
    gd = G.GpuProblem("hyperFS", 4, 4, resource=DET)
    assert not ga.ceed.is_deterministic
    ga.residual(); gd.residual()
    x = np.random.default_rng(9).standard_normal(ga.mesh.lsize(4))
    assert rel_err(ga.jacobian(2, x), gd.jacobian(2, x)) < 1e-14


@pytest.mark.parametrize("p", [3, 4])
def test_deterministic_prolongation_on_a_reoriented_mesh_is_the_ordered_sum(p):
    """Prolong_Ceed in deterministic mode on a mesh with mixed element orientation: within 1e-12 of the oracle, and
    bit for bit the sum, per fine dof in ascending (element, node) order, of the element interpolants of one d_evec
    run scaled by the inverse multiplicity.  An injected prolongation (each holder stores its own copy, the last
    store wins) does not give that sum: the copies of differently oriented elements differ in the last bit."""
    import torch
    import gpu_helpers as G
    from ceedpetscsolid_b200 import matops
    from ceedpetscsolid_b200.ceed import b2, lib
    from ceedpetscsolid_b200.exodus import tube_mesh
    from helpers import reoriented
    from oracle import oracle
    mesh = reoriented(tube_mesh(2, 6, 2), seed=5)
    g = G.GpuProblem("hyperFS", None, p, multigrid="uniform", mesh=mesh, resource=DET)
    dms = [matops.LevelDM(mesh, deg, bc_faces=None) for deg in g.degrees]
    users = [matops.setup_jacobian_ctx(dms[l], g.ceed, g.data[l], g.phys) for l in range(len(g.degrees))]
    rng = np.random.default_rng(p)
    for level in range(1, len(g.degrees)):
        pc, pf = g.degrees[level - 1], g.degrees[level]
        Pf3, nelem = (pf + 1) ** 3, mesh.nelem
        offc, offf = mesh.offsets(pc), mesh.offsets(pf)
        lc, lf = mesh.lsize(pc), mesh.lsize(pf)
        ctx = matops.setup_prolong_restrict_ctx(dms[level - 1], dms[level], g.ceed, g.data[level - 1], g.data[level],
                                                users[level - 1], users[level])
        assert ctx.fusedScale is not None and not ctx.inject
        xc = rng.standard_normal(lc)
        Xc, Yf = torch.from_numpy(xc).cuda(), dms[level].create_global_vector()
        ctx.locVecF.fill_(123.0)
        matops.Prolong_Ceed(ctx, Xc, Yf)
        got = Yf.cpu().numpy()
        minv = 1.0 / oracle.multiplicity(nelem, Pf3, 3, lf, offf)
        ref = oracle.transfer(False, nelem, pc + 1, pf + 1, offc, offf, xc, lf) * minv
        assert np.abs(got - ref).max() <= TOL * np.abs(ref).max()
        # host reference from one d_evec run of the same kernel and basis, no scaling inside
        J = np.ascontiguousarray(g.data[level].basisCtoF.interp1d)
        d_offc = torch.from_numpy(offc.reshape(-1)).cuda()
        d_offf = torch.from_numpy(offf.reshape(-1)).cuda()
        ev = torch.full((nelem * Pf3 * 3,), np.nan, dtype=torch.float64, device="cuda")
        scratch = torch.zeros(lf, dtype=torch.float64, device="cuda")
        b2(lib.b200_apply_transfer(0, nelem, pc + 1, pf + 1, J.ctypes.data, d_offc.data_ptr(), d_offf.data_ptr(), None,
                                   0, Xc.data_ptr(), scratch.data_ptr(), ev.data_ptr()))
        torch.cuda.synchronize()
        dof = (offf.reshape(-1, 1) + np.arange(3)).reshape(-1)
        vals = ev.cpu().numpy() * minv[dof]
        order = np.argsort(dof, kind="stable")                   # ascending (element, node) within every dof
        d, v = dof[order], vals[order]
        rank = np.arange(d.size) - np.searchsorted(d, d, side="left")
        host = np.zeros(lf)
        for k in range(int(rank.max()) + 1):
            host[d[rank == k]] += v[rank == k]
        assert np.array_equal(got.view(np.uint64), host.view(np.uint64)), (
            f"({pc + 1}, {pf + 1}): {np.count_nonzero(got != host)} of {lf} dofs differ from the ordered sum")
