"""Parity of the /gpu/b200 CUDA path against the CPU oracle, through the libCEED C API
(libceed_b200.so).  FP64; tolerance from BASELINE.json north_star: 1e-12 relative."""
import numpy as np
import pytest

from helpers import OracleProblem, rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-12


@pytest.fixture(scope="module")
def G():
    import gpu_helpers
    return gpu_helpers


CASES = [  # problem, n, p, qextra, perm      (("linElas", 8, 2): BASELINE configs[0] = C1 exactly)
    ("linElas", 3, 1, 0, None), ("linElas", 4, 2, 0, None), ("linElas", 8, 2, 0, None), ("linElas", 3, 3, 0, 11),
    ("hyperSS", 3, 2, 0, None), ("hyperSS", 4, 3, 0, None), ("hyperSS", 2, 4, 0, 12),
    ("hyperFS", 3, 2, 0, None), ("hyperFS", 3, 3, 0, None), ("hyperFS", 3, 4, 0, None),
    ("hyperFS", 2, 4, 1, None), ("hyperFS", 2, 2, 1, 13), ("hyperFS", (7, 2, 3), 4, 0, None),
]


@pytest.mark.parametrize("problem,n,p,qextra,perm", CASES)
def test_setupgeo_residual_jacobian_diagonal(G, problem, n, p, qextra, perm):
    g = G.GpuProblem(problem, n, p, qextra=qextra, node_perm_seed=perm)
    o = OracleProblem(problem, n, p, qextra=qextra)
    # geometric factors (generic path: restriction + basis + SetupGeo kernels)
    qd = g.strided_to_plain(g.fine.Erestrictqdi, g.fine.qdata)
    assert rel_err(qd, o.qdata) < TOL
    # residual (fused) and the gradu it stores
    yo = o.residual_fine(o.u_fine)
    yg = g.residual()
    if perm is not None:
        tmp = np.empty_like(yo).reshape(-1, 3); tmp[g.perm] = yo.reshape(-1, 3); yo = tmp.reshape(-1)
    fused_expected = (p + 1 + qextra) <= 5  # fused kernels are instantiated for Q <= 5
    assert g.fine.opApply.is_fused == fused_expected
    assert rel_err(yg, yo) < TOL
    if o.has_gradu:
        gu = g.strided_to_plain(g.fine.ErestrictGradui, g.fine.gradu)
        assert rel_err(gu, o.gradu) < TOL
    # Jacobian on every p-multigrid level (all levels stream the fine quadrature data)
    rng = np.random.default_rng(1)
    for level, deg in enumerate(g.degrees):
        ol = OracleProblem(problem, n, p, pl=deg, qextra=qextra)
        x = rng.standard_normal(ol.lsize)
        yo = ol.jacobian(x)
        do = ol.diagonal()
        xg = x
        if perm is not None and level == len(g.degrees) - 1:
            def P(v):
                t = np.empty_like(v).reshape(-1, 3); t[g.perm] = v.reshape(-1, 3); return t.reshape(-1)
            xg, yo, do = P(x), P(yo), P(do)
        assert g.data[level].opJacob.is_fused == fused_expected
        assert rel_err(g.jacobian(level, xg), yo) < TOL, (level, deg)
        assert rel_err(g.diagonal(level), do) < TOL, (level, deg)


def test_jacobian_tracks_new_linearisation_point(G):
    """gradu rewritten by a residual evaluation invalidates the Jacobian cache."""
    g = G.GpuProblem("hyperFS", 3, 2)
    o = OracleProblem("hyperFS", 3, 2)
    x = np.random.default_rng(2).standard_normal(o.lsize)
    g.residual()
    y1 = g.jacobian(len(g.degrees) - 1, x)
    u2 = 1.7 * o.u_fine
    o.residual_fine(u2)
    g.residual(u2)
    y2 = g.jacobian(len(g.degrees) - 1, x)
    assert rel_err(y2, o.jacobian(x)) < TOL
    assert rel_err(y2, y1) > 1e-6


def test_generic_path_operator_matches_fused(G):
    """(P,Q) = (4,6) is not instantiated as a fused kernel -> restriction/basis/QFunction kernels."""
    g = G.GpuProblem("hyperFS", 2, 3, qextra=2, multigrid="none")
    o = OracleProblem("hyperFS", 2, 3, qextra=2)
    assert not g.fine.opApply.is_fused and not g.data[-1].opJacob.is_fused
    assert rel_err(g.residual(), o.residual_fine(o.u_fine)) < TOL
    x = np.random.default_rng(3).standard_normal(o.lsize)
    assert rel_err(g.jacobian(0, x), o.jacobian(x)) < TOL


def test_transfer_operators_and_multiplicity(G):
    from oracle import oracle
    g = G.GpuProblem("hyperFS", 3, 4)
    rng = np.random.default_rng(4)
    for level in range(1, len(g.degrees)):
        pc, pf = g.degrees[level - 1], g.degrees[level]
        offc, offf = g.mesh.offsets(pc), g.mesh.offsets(pf)
        lc, lf = g.mesh.lsize(pc), g.mesh.lsize(pf)
        c, f = rng.standard_normal(lc), rng.standard_normal(lf)
        d = g.data[level]
        assert d.opProlong.is_fused and d.opRestrict.is_fused
        assert rel_err(g.apply(d.opProlong, c, lf), oracle.transfer(False, g.mesh.nelem, pc + 1, pf + 1, offc, offf, c, lf)) < TOL
        assert rel_err(g.apply(d.opRestrict, f, lc), oracle.transfer(True, g.mesh.nelem, pc + 1, pf + 1, offc, offf, f, lc)) < TOL
        m = d.Erestrictu.create_vector()
        d.Erestrictu.get_multiplicity(m)
        np.testing.assert_array_equal(m.to_numpy(), oracle.multiplicity(g.mesh.nelem, (pf + 1) ** 3, 3, lf, offf))


def test_matshell_callbacks_device_and_host_memtype(G):
    """ApplyJacobian_Ceed / FormResidual_Ceed / GetDiag_Ceed through UserMult, both memtypes."""
    import torch
    from ceedpetscsolid_b200 import matops
    from ceedpetscsolid_b200.ceed import MEM_DEVICE, MEM_HOST
    g = G.GpuProblem("hyperFS", 3, 2)
    o = OracleProblem("hyperFS", 3, 2)
    g.residual()
    lvl = len(g.degrees) - 1
    dm = matops.LevelDM(g.mesh, g.degrees[lvl], bc_faces="all")
    free = ~np.repeat(dm.bc_nodes, 3)
    xg = np.random.default_rng(5).standard_normal(dm.nglobal)
    xl = np.zeros(o.lsize); xl[free] = xg
    yref = o.jacobian(xl)[free]
    dref = o.diagonal()[free]
    for mem in (MEM_DEVICE, MEM_HOST):
        user = matops.setup_jacobian_ctx(dm, g.ceed, g.data[lvl], g.phys, memType=mem)
        X = dm.create_global_vector(mem); Y = dm.create_global_vector(mem); D = dm.create_global_vector(mem)
        X.copy_(torch.from_numpy(xg))
        matops.ApplyJacobian_Ceed(user, X, Y)
        matops.GetDiag_Ceed(user, D)
        torch.cuda.synchronize()
        assert rel_err(Y.cpu().numpy(), yref) < TOL
        assert rel_err(D.cpu().numpy(), dref) < TOL
        assert float(user.Xloc.abs().max()) == 0.0  # GetDiag_Ceed re-zeroes Xloc (matops.c:241)


def test_errors_are_loud(G):
    from ceedpetscsolid_b200 import ceed as libceed
    c = libceed.Ceed("/gpu/b200")
    with pytest.raises(libceed.CeedError):
        libceed.Ceed("/cpu/self")
    qf = c.QFunction(1, "somewhere/user.h:NotAKnownQFunction")
    qf.add_input("u", 1, libceed.EVAL_NONE)
    qf.add_output("v", 1, libceed.EVAL_NONE)
    r = c.StridedElemRestriction(2, 8, 1, 16)
    op = c.Operator(qf)
    op.set_field("u", r, libceed.BASIS_COLLOCATED, libceed.VECTOR_ACTIVE)
    op.set_field("v", r, libceed.BASIS_COLLOCATED, libceed.VECTOR_ACTIVE)
    u, v = c.Vector(16), c.Vector(16)
    u.set_value(1.0)
    with pytest.raises(libceed.CeedError, match="no CPU fallback"):
        op.apply(u, v)
    with pytest.raises(libceed.CeedError):
        c.ElemRestriction(1, 8, 3, 1, 10, np.arange(8) * 3)  # offsets out of range


@pytest.mark.parametrize("masked", [False, True])
def test_prolong_restrict_with_scaling_inside_the_kernel(G, masked):
    """Prolong_Ceed / Restrict_Ceed (matops.c:115-203): the fused transfer kernels apply the inverse multiplicity
    themselves (CeedOperatorSetTransferScalingB200; the prolongation stores the interpolant) -- same result as the
    reference sequence  operator apply + VecPointwiseMult  and as the oracle."""
    import torch
    from ceedpetscsolid_b200 import matops
    from oracle import oracle
    g = G.GpuProblem("hyperFS", (3, 4, 2), 4)
    rng = np.random.default_rng(6)
    dms = [matops.LevelDM(g.mesh, deg, bc_faces="all", masked=masked) for deg in g.degrees]
    users = [matops.setup_jacobian_ctx(dms[l], g.ceed, g.data[l], g.phys) for l in range(len(g.degrees))]
    for level in range(1, len(g.degrees)):
        pc, pf = g.degrees[level - 1], g.degrees[level]
        dmC, dmF = dms[level - 1], dms[level]
        plain = matops.setup_prolong_restrict_ctx(dmC, dmF, g.ceed, g.data[level - 1], g.data[level], users[level - 1],
                                                  users[level], fuse_scaling=False)
        Xc, Xf = dmC.create_global_vector(), dmF.create_global_vector()
        Xc.copy_(torch.from_numpy(rng.standard_normal(dmC.nglobal))); dmC.zero_constrained(Xc)
        Xf.copy_(torch.from_numpy(rng.standard_normal(dmF.nglobal))); dmF.zero_constrained(Xf)
        Yf0, Yc0 = dmF.create_global_vector(), dmC.create_global_vector()
        assert plain.fusedScale is None
        matops.Prolong_Ceed(plain, Xc, Yf0)
        matops.Restrict_Ceed(plain, Xf, Yc0)
        fused = matops.setup_prolong_restrict_ctx(dmC, dmF, g.ceed, g.data[level - 1], g.data[level], users[level - 1],
                                                  users[level])
        assert fused.fusedScale is not None and fused.inject
        Yf1, Yc1 = dmF.create_global_vector(), dmC.create_global_vector()
        fused.locVecF.fill_(123.0)   # injected prolongation needs no zeroed work vector
        matops.Prolong_Ceed(fused, Xc, Yf1)
        matops.Restrict_Ceed(fused, Xf, Yc1)
        torch.cuda.synchronize()
        assert rel_err(Yf1.cpu().numpy(), Yf0.cpu().numpy()) < TOL
        assert rel_err(Yc1.cpu().numpy(), Yc0.cpu().numpy()) < TOL
        # oracle: interpolate the coarse L-vector, scale by the inverse multiplicity
        offc, offf = g.mesh.offsets(pc), g.mesh.offsets(pf)
        lc, lf = g.mesh.lsize(pc), g.mesh.lsize(pf)
        xc_l = np.zeros(lc)
        freeC, freeF = ~np.repeat(dmC.bc_nodes, 3), ~np.repeat(dmF.bc_nodes, 3)
        xc_l[freeC] = Xc.cpu().numpy()[freeC] if masked else Xc.cpu().numpy()
        mult = oracle.multiplicity(g.mesh.nelem, (pf + 1) ** 3, 3, lf, offf)
        yo = oracle.transfer(False, g.mesh.nelem, pc + 1, pf + 1, offc, offf, xc_l, lf) / mult
        got = Yf1.cpu().numpy()
        assert rel_err(got[freeF] if masked else got, yo[freeF]) < TOL
        # plain operator semantics are restored when the scaling is removed
        g.data[level].opProlong.set_transfer_scaling(None)
        g.data[level].opRestrict.set_transfer_scaling(None)
        c = rng.standard_normal(lc)
        assert rel_err(g.apply(g.data[level].opProlong, c, lf), oracle.transfer(False, g.mesh.nelem, pc + 1, pf + 1, offc, offf, c, lf)) < TOL


def max_rel(got, ref):
    return np.abs(np.asarray(got) - ref).max() / np.abs(ref).max()


@pytest.mark.parametrize("resource", ["/gpu/b200", "/gpu/b200:deterministic"], ids=["default", "deterministic"])
@pytest.mark.parametrize("problem,p", [("linElas", 4), ("hyperSS", 4), ("hyperFS", 4), ("hyperFS", 3)])
def test_reoriented_tube_every_level_and_transfer(G, resource, problem, p):
    """a tube whose elements are listed under random cube rotations (neighbours with different local axes), uniform
    p-multigrid: every level's Jacobian and diagonal, both transfers between every pair of levels -- at degree 4 the
    pairs (2,5), (3,5), (4,5), (5,5) and the transfers (2,3), (3,4), (4,5) -- against the oracle, elementwise"""
    from oracle import oracle
    from ceedpetscsolid_b200.exodus import tube_mesh
    from helpers import reoriented
    mesh = reoriented(tube_mesh(2, 6, 2), seed=5)
    g = G.GpuProblem(problem, None, p, multigrid="uniform", mesh=mesh, resource=resource)
    assert g.degrees == list(range(1, p + 1))
    o = OracleProblem(problem, None, p, mesh=mesh)
    assert max_rel(g.residual(), o.residual_fine(o.u_fine)) < TOL
    rng = np.random.default_rng(p)
    for level, deg in enumerate(g.degrees):
        ol = OracleProblem(problem, None, p, pl=deg, mesh=mesh)
        assert g.data[level].opJacob.is_fused
        x = rng.standard_normal(ol.lsize)
        assert max_rel(g.jacobian(level, x), ol.jacobian(x)) < TOL, (level, deg)
        assert max_rel(g.diagonal(level), ol.diagonal()) < TOL, (level, deg)
        if level == 0:
            continue
        pc, pf = g.degrees[level - 1], deg
        offc, offf = mesh.offsets(pc), mesh.offsets(pf)
        lc, lf = mesh.lsize(pc), mesh.lsize(pf)
        c, f = rng.standard_normal(lc), rng.standard_normal(lf)
        d = g.data[level]
        assert d.opProlong.is_fused and d.opRestrict.is_fused
        assert max_rel(g.apply(d.opProlong, c, lf), oracle.transfer(False, mesh.nelem, pc + 1, pf + 1, offc, offf, c, lf)) < TOL
        assert max_rel(g.apply(d.opRestrict, f, lc), oracle.transfer(True, mesh.nelem, pc + 1, pf + 1, offc, offf, f, lc)) < TOL
