"""The reference's OWN host code on /gpu/b200.

oracle/_ref/ref_driver (built by `make -C oracle refdriver` where /root/reference is mounted; the binary travels to
the GPU box) links the reference's src/setuplibceed.c, src/matops.c and src/misc.c -- compiled unchanged, nothing
copied -- against this repository's <ceed.h> / libceed_b200.so and a functional miniature of the PETSc calls they make
(tests/c/petsc_mini).  The reference's SetupLibceedFineLevel / SetupLibceedLevel build every libCEED object (with the
reference's own QFunction pointers: the backend's QFunction guard runs on them), SetupJacobianCtx /
SetupProlongRestrictCtx wire the MatShell contexts, and FormResidual_Ceed, ApplyJacobian_Ceed, GetDiag_Ceed,
Prolong_Ceed, Restrict_Ceed, ComputeStrainEnergy and ViewDiagnosticQuantities are the reference's functions.  This test writes the mesh
(closure indices with essential-BC dofs encoded as -(loc+1), as DMPlex hands them to CreateRestrictionPlex) and
the vectors, runs the driver with host and with device memtype, and compares every output with the CPU oracle.
"""
import os

import pytest

from ref_host_code import DRIVER, GOLDEN_CASES, ROOT, TOL, run_and_check


@pytest.mark.gpu
@pytest.mark.parametrize("resource", ["/gpu/b200", "/gpu/b200:deterministic"])
@pytest.mark.parametrize("memtype", [0, 1], ids=["memtype_host", "memtype_device"])
@pytest.mark.parametrize("problem,n,degrees", [("hyperFS", (3, 2, 2), [1, 2, 4]), ("hyperSS", (2, 2, 3), [1, 2, 3]),
                                               ("linElas", (3, 3, 2), [1, 2])])
def test_reference_setup_and_matshell_callbacks_drive_the_backend(tmp_path, problem, n, degrees, memtype, resource):
    if not os.path.exists(DRIVER):
        pytest.skip("oracle/_ref/ref_driver not built (needs /root/reference at build time)")
    run_and_check(DRIVER, tmp_path, problem, n, degrees, memtype, resource)


@pytest.mark.gpu
@pytest.mark.parametrize("resource", ["/gpu/b200", "/gpu/b200:deterministic"])
@pytest.mark.parametrize("problem,n,degrees", GOLDEN_CASES)
def test_matshell_callbacks_on_the_backend_reproduce_the_committed_output_of_the_reference_host_code(problem, n, degrees,
                                                                                                     resource):
    """no driver, no reference tree: the seeded cases of the driver through this package's restatement of the reference's
    set-up and MatShell callbacks (setuplibceed.py, matops.py) on /gpu/b200, piece by piece against what the reference's
    host code and QFunctions wrote on the CPU (tests/golden/ref_host_code_golden.npz)"""
    import numpy as np
    import torch
    from ceedpetscsolid_b200 import ceed as libceed
    from ceedpetscsolid_b200 import matops, setuplibceed
    from helpers import rel_err
    from ref_host_code import GOLDEN, case_key, make_case, split_like

    o, _, xs = make_case(problem, n, degrees)
    mesh, p = o.mesh, degrees[-1]
    ceed = libceed.Ceed(resource)
    levels, data, phys = setuplibceed.setup_all(ceed, mesh, problem, p)
    assert levels == degrees
    dms = [matops.LevelDM(mesh, deg, bc_faces="all") for deg in degrees]     # compressed global vectors: the free dofs
    users = [matops.setup_jacobian_ctx(dms[l], ceed, data[l], phys) for l in range(len(degrees))]
    fu, fine = users[-1], data[-1]
    u = torch.from_numpy(o.u_fine).cuda()
    bc_values = u[dms[-1].bc_idx.long()].contiguous()
    res = matops.UserMult(dm=fu.dm, Xloc=fu.Xloc, Yloc=fu.Yloc, Xceed=fu.Xceed, Yceed=fu.Yceed, op=fine.opApply,
                          qf=fine.qfApply, ceed=ceed, phys=phys, bc_values=lambda load: bc_values)
    state = u[dms[-1].free_owned_idx.long()].contiguous()

    def out(dm, fn):
        y = dm.create_global_vector()
        fn(y)
        return y.cpu().numpy()

    def dev(a):
        return torch.from_numpy(a).cuda()
    # in the driver's order: residual (writes gradu), Jacobian and diagonal per level, transfers, energy, diagnostics
    parts = [("residual", out(dms[-1], lambda y: matops.FormResidual_Ceed(state, y, res)))]
    for l, deg in enumerate(degrees):
        parts.append((f"jacobian p={deg}", out(dms[l], lambda y: matops.ApplyJacobian_Ceed(users[l], dev(xs[l]), y))))
        parts.append((f"diagonal p={deg}", out(dms[l], lambda y: matops.GetDiag_Ceed(users[l], y))))
    for l in range(1, len(degrees)):
        ctx = matops.setup_prolong_restrict_ctx(dms[l - 1], dms[l], ceed, data[l - 1], data[l], users[l - 1], users[l])
        parts.append((f"prolong {degrees[l - 1]}->{degrees[l]}",
                      out(dms[l], lambda y: matops.Prolong_Ceed(ctx, dev(xs[l - 1]), y))))
        parts.append((f"restrict {degrees[l]}->{degrees[l - 1]}",
                      out(dms[l - 1], lambda y: matops.Restrict_Ceed(ctx, dev(xs[l]), y))))
    setuplibceed.setup_energy(ceed, mesh, problem, fine, phys)
    setuplibceed.setup_diagnostic(ceed, mesh, problem, fine, phys)
    parts.append(("strain energy", np.array([matops.ComputeStrainEnergy(res, fine.opEnergy, state)])))
    diag = matops.ComputeDiagnosticQuantities(res, fine.opDiagnostic, fine.ErestrictDiagnostic, state).cpu().numpy()
    parts += [(f"diagnostic column {k}", diag[:, k]) for k in range(8)]
    with np.load(GOLDEN) as g:
        want = g[case_key(problem, n, degrees)]
    for (name, got), ref in zip(parts, split_like(want, parts, mesh.num_nodes(p))):
        assert got.shape == ref.shape and rel_err(got, ref) < TOL, name


def test_driver_sources_exist_and_build_recipe_names_the_reference_files():
    """CPU-side sanity: the recipe compiles the reference files where they lie and nothing of them is in this repo"""
    mk = open(os.path.join(ROOT, "oracle", "Makefile")).read()
    for f in ("setuplibceed.c", "matops.c", "misc.c"):
        assert f"$(REF)/src/{f}" in mk
        assert not os.path.exists(os.path.join(ROOT, "tests", "c", f))
    assert os.path.exists(os.path.join(ROOT, "tests", "c", "ref_driver.c"))
    assert os.path.exists(os.path.join(ROOT, "tests", "c", "petsc_mini", "petsc_mini.c"))
