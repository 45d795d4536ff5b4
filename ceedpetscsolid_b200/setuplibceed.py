"""Build the libCEED objects of the solid-mechanics mini-app on the `/gpu/b200` backend.

Mirrors, call for call, what the reference does in
/root/reference/src/setuplibceed.c:
  problemOptions[]          :41-107   -> PROBLEM_OPTIONS
  CreateRestrictionPlex     :194-240  -> create_restriction (offsets come from mesh.BoxMesh)
  SetupLibceedFineLevel     :243-745  -> setup_fine_level   (restrictions, bases, qdata via the
                                        SetupGeo operator, residual operator opApply)
  SetupLibceedLevel         :748-939  -> setup_level        (per-level Jacobian operator,
                                        prolongation / restriction operators)
with the same field names, eval modes, sizes and QFunction source locators, so that the
operator objects the backend sees are the ones the reference would hand to it.
"""
from dataclasses import dataclass, field

from . import ceed as libceed
from .ceed import (BASIS_COLLOCATED, ELEMRESTRICTION_NONE, EVAL_GRAD, EVAL_INTERP, EVAL_NONE, EVAL_WEIGHT, GAUSS,
                   GAUSS_LOBATTO, VECTOR_ACTIVE, VECTOR_NONE, Physics)

# problemOptions[] (setuplibceed.c:41-107): qdatasize, residual / Jacobian QFunction locators
PROBLEM_OPTIONS = {
    "linElas": dict(qdatasize=10, setupgeo="qfunctions/common.h:SetupGeo", apply="qfunctions/linElas.h:LinElasF",
                    jacob="qfunctions/linElas.h:LinElasdF", qmode=GAUSS, nonlinear=False,
                    energy="qfunctions/linElas.h:LinElasEnergy", diagnostic="qfunctions/linElas.h:LinElasDiagnostic"),
    "hyperSS": dict(qdatasize=10, setupgeo="qfunctions/common.h:SetupGeo", apply="qfunctions/hyperSS.h:HyperSSF",
                    jacob="qfunctions/hyperSS.h:HyperSSdF", qmode=GAUSS, nonlinear=True,
                    energy="qfunctions/hyperSS.h:HyperSSEnergy", diagnostic="qfunctions/hyperSS.h:HyperSSDiagnostic"),
    "hyperFS": dict(qdatasize=10, setupgeo="qfunctions/common.h:SetupGeo", apply="qfunctions/hyperFS.h:HyperFSF",
                    jacob="qfunctions/hyperFS.h:HyperFSdF", qmode=GAUSS, nonlinear=True,
                    energy="qfunctions/hyperFS.h:HyperFSEnergy", diagnostic="qfunctions/hyperFS.h:HyperFSDiagnostic"),
}


def level_degrees(degree, multigrid="logarithmic"):
    """Level schedule of /root/reference/src/cloptions.c:195-225."""
    if multigrid == "none" or degree == 1:
        return [degree]
    if multigrid == "uniform":
        return list(range(1, degree + 1))
    levels, d = [], 1
    while d < degree:
        levels.append(d)
        d *= 2
    return levels + [degree]


@dataclass
class CeedData:
    """elasticity.h:218-240 CeedData (per level)."""
    basisx: object = None
    basisu: object = None
    basisCtoF: object = None
    Erestrictx: object = None
    Erestrictu: object = None
    Erestrictqdi: object = None
    ErestrictGradui: object = None
    qfApply: object = None
    qfJacob: object = None
    opApply: object = None
    opJacob: object = None
    opRestrict: object = None
    opProlong: object = None
    qdata: object = None
    gradu: object = None
    xceed: object = None
    yceed: object = None
    # post-processing (setuplibceed.c:645-737)
    ErestrictEnergy: object = None
    basisEnergy: object = None
    qfEnergy: object = None
    opEnergy: object = None
    ErestrictDiagnostic: object = None
    ErestrictqdDiagnostici: object = None
    basisDiagnostic: object = None
    qdataDiagnostic: object = None
    qfDiagnostic: object = None
    opDiagnostic: object = None
    keep: list = field(default_factory=list)


def create_restriction(ceed, mesh, P, ncomp, node_perm=None):
    """CreateRestrictionPlex (setuplibceed.c:194-240): one offset per element node = dof of
    component 0, compstride 1 (interlaced), lsize = local vector size."""
    off = mesh.offsets(P - 1, ncomp=ncomp, node_perm=node_perm)
    return ceed.ElemRestriction(mesh.nelem, P ** 3, ncomp, 1, ncomp * mesh.num_nodes(P - 1), off)


def problem_options(problem, qf_locators=None):
    """PROBLEM_OPTIONS[problem] with the residual ("apply") and Jacobian ("jacob") QFunction locators replaced by those
    of qf_locators.  The problem still decides the field layout; a locator the backend has no built-in body for needs
    the "/gpu/b200:jit" resource, which compiles it from its "<file>:<Name>" source."""
    opt = dict(PROBLEM_OPTIONS[problem])
    if qf_locators:
        unknown = set(qf_locators) - {"apply", "jacob"}
        if unknown:
            raise ValueError(f"qf_locators: only 'apply' and 'jacob' can be replaced (got {sorted(unknown)})")
        opt.update(qf_locators)
    return opt


def setup_fine_level(ceed, mesh, problem, degree, phys, data, qextra=0, node_perm=None, qf_locators=None):
    """SetupLibceedFineLevel (setuplibceed.c:243-545, the parts on the hot path)."""
    opt = problem_options(problem, qf_locators)
    P, Q = degree + 1, degree + 1 + qextra
    dim = ncompx = ncompu = 3
    qdatasize = opt["qdatasize"]
    nelem = mesh.nelem
    d = data
    # -- restrictions (:279-318)
    d.Erestrictx = create_restriction(ceed, mesh, 2, ncompx)
    d.Erestrictu = create_restriction(ceed, mesh, P, ncompu, node_perm)
    d.Erestrictqdi = ceed.StridedElemRestriction(nelem, Q ** 3, qdatasize, qdatasize * nelem * Q ** 3)
    if opt["nonlinear"]:
        d.ErestrictGradui = ceed.StridedElemRestriction(nelem, Q ** 3, dim * ncompu, dim * ncompu * nelem * Q ** 3)
    # -- element coordinates (:323-329): HOST array, COPY_VALUES
    xcoord = d.Erestrictx.create_vector()
    xcoord.set_array(mesh.coord_lvector(), libceed.MEM_HOST, libceed.COPY_VALUES)
    # -- bases (:335-341)
    d.basisu = ceed.BasisTensorH1Lagrange(dim, ncompu, P, Q, opt["qmode"])
    d.basisx = ceed.BasisTensorH1Lagrange(dim, ncompx, 2, Q, opt["qmode"])
    # -- persistent vectors (:353-361)
    nqpts = d.basisu.num_qpts
    d.qdata = ceed.Vector(qdatasize * nelem * nqpts)
    if opt["nonlinear"]:
        d.gradu = ceed.Vector(dim * ncompu * nelem * nqpts)
    # -- geometric factors (:370-393)
    qfSetupGeo = ceed.QFunction(1, opt["setupgeo"])
    qfSetupGeo.add_input("dx", ncompx * dim, EVAL_GRAD)
    qfSetupGeo.add_input("weight", 1, EVAL_WEIGHT)
    qfSetupGeo.add_output("qdata", qdatasize, EVAL_NONE)
    opSetupGeo = ceed.Operator(qfSetupGeo)
    opSetupGeo.set_field("dx", d.Erestrictx, d.basisx, VECTOR_ACTIVE)
    opSetupGeo.set_field("weight", ELEMRESTRICTION_NONE, d.basisx, VECTOR_NONE)
    opSetupGeo.set_field("qdata", d.Erestrictqdi, BASIS_COLLOCATED, VECTOR_ACTIVE)
    opSetupGeo.apply(xcoord, d.qdata)
    qfSetupGeo.destroy()
    opSetupGeo.destroy()
    xcoord.destroy()
    # -- residual evaluator (:518-542)
    d.qfApply = ceed.QFunction(1, opt["apply"])
    d.qfApply.add_input("du", ncompu * dim, EVAL_GRAD)
    d.qfApply.add_input("qdata", qdatasize, EVAL_NONE)
    d.qfApply.add_output("dv", ncompu * dim, EVAL_GRAD)
    if opt["nonlinear"]:
        d.qfApply.add_output("gradu", ncompu * dim, EVAL_NONE)
    d.qfApply.set_context(phys)
    d.opApply = ceed.Operator(d.qfApply)
    d.opApply.set_field("du", d.Erestrictu, d.basisu, VECTOR_ACTIVE)
    d.opApply.set_field("qdata", d.Erestrictqdi, BASIS_COLLOCATED, d.qdata)
    d.opApply.set_field("dv", d.Erestrictu, d.basisu, VECTOR_ACTIVE)
    if opt["nonlinear"]:
        # the reference passes basisu here although the mode is EVAL_NONE (:538-539)
        d.opApply.set_field("gradu", d.ErestrictGradui, d.basisu, d.gradu)
    return d


FORCING_OPTIONS = {  # forcingOptions[] (setuplibceed.c:110-125)
    "constant": "qfunctions/constantForce.h:SetupConstantForce",
    "mms": "qfunctions/manufacturedForce.h:SetupMMSForce",
}


def setup_forcing(ceed, mesh, data, forcing, phys, forcing_vector, force_ceed):
    """Forcing term (setuplibceed.c:550-584): force_L = E^T B^T f(B x, qdata)."""
    import ctypes as C
    d = data
    qf = ceed.QFunction(1, FORCING_OPTIONS[forcing])
    qf.add_input("x", 3, EVAL_INTERP)
    qf.add_input("qdata", 10, EVAL_NONE)
    qf.add_output("force", 3, EVAL_INTERP)
    if forcing == "mms":
        qf.set_context(phys)
    else:
        fv = (C.c_double * 3)(*forcing_vector)
        qf.set_context(fv, size=8)  # sizeof(*appCtx->forcingVector), setuplibceed.c:566-567
    xcoord = d.Erestrictx.create_vector()
    xcoord.set_array(mesh.coord_lvector(), libceed.MEM_HOST, libceed.COPY_VALUES)
    op = ceed.Operator(qf)
    op.set_field("x", d.Erestrictx, d.basisx, VECTOR_ACTIVE)
    op.set_field("qdata", d.Erestrictqdi, BASIS_COLLOCATED, d.qdata)
    op.set_field("force", d.Erestrictu, d.basisu, VECTOR_ACTIVE)
    op.apply(xcoord, force_ceed)
    op.destroy(); qf.destroy(); xcoord.destroy()


def setup_energy(ceed, mesh, problem, data, phys, node_perm=None):
    """Strain-energy operator (setuplibceed.c:645-670): energy_L = E_e^T B_e^T [ w detJ psi(grad u) ], one scalar dof per
    mesh node (dmEnergy, ncompe = 1); ComputeStrainEnergy sums the entries."""
    d, opt = data, PROBLEM_OPTIONS[problem]
    P, Q = d.basisu.P, d.basisu.Q
    d.ErestrictEnergy = create_restriction(ceed, mesh, P, 1, node_perm)
    d.basisEnergy = ceed.BasisTensorH1Lagrange(3, 1, P, Q, opt["qmode"])
    d.qfEnergy = ceed.QFunction(1, opt["energy"])
    d.qfEnergy.add_input("du", 9, EVAL_GRAD)
    d.qfEnergy.add_input("qdata", opt["qdatasize"], EVAL_NONE)
    d.qfEnergy.add_output("energy", 1, EVAL_INTERP)
    d.qfEnergy.set_context(phys)
    d.opEnergy = ceed.Operator(d.qfEnergy)
    d.opEnergy.set_field("du", d.Erestrictu, d.basisu, VECTOR_ACTIVE)
    d.opEnergy.set_field("qdata", d.Erestrictqdi, BASIS_COLLOCATED, d.qdata)
    d.opEnergy.set_field("energy", d.ErestrictEnergy, d.basisEnergy, VECTOR_ACTIVE)
    return d.opEnergy


def setup_diagnostic(ceed, mesh, problem, data, phys, node_perm=None):
    """Nodal diagnostic operator (setuplibceed.c:672-737): geometric factors collocated at the GLL nodes
    (basis P -> P, CEED_GAUSS_LOBATTO), then (u, grad u, qdata) -> 8 values per node, EVAL_NONE out."""
    d, opt = data, PROBLEM_OPTIONS[problem]
    P = d.basisu.P
    nelem, qdatasize = mesh.nelem, opt["qdatasize"]
    d.ErestrictDiagnostic = create_restriction(ceed, mesh, P, 8, node_perm)
    d.ErestrictqdDiagnostici = ceed.StridedElemRestriction(nelem, P ** 3, qdatasize, qdatasize * nelem * P ** 3)
    d.basisDiagnostic = ceed.BasisTensorH1Lagrange(3, 3, P, P, GAUSS_LOBATTO)
    d.qdataDiagnostic = ceed.Vector(qdatasize * nelem * P ** 3)
    basisx = ceed.BasisTensorH1Lagrange(3, 3, 2, P, GAUSS_LOBATTO)
    qfSetupGeo = ceed.QFunction(1, opt["setupgeo"])
    qfSetupGeo.add_input("dx", 9, EVAL_GRAD)
    qfSetupGeo.add_input("weight", 1, EVAL_WEIGHT)
    qfSetupGeo.add_output("qdata", qdatasize, EVAL_NONE)
    opSetupGeo = ceed.Operator(qfSetupGeo)
    opSetupGeo.set_field("dx", d.Erestrictx, basisx, VECTOR_ACTIVE)
    opSetupGeo.set_field("weight", ELEMRESTRICTION_NONE, basisx, VECTOR_NONE)
    opSetupGeo.set_field("qdata", d.ErestrictqdDiagnostici, BASIS_COLLOCATED, VECTOR_ACTIVE)
    xcoord = d.Erestrictx.create_vector()
    xcoord.set_array(mesh.coord_lvector(), libceed.MEM_HOST, libceed.COPY_VALUES)
    opSetupGeo.apply(xcoord, d.qdataDiagnostic)
    for o in (basisx, qfSetupGeo, opSetupGeo, xcoord):
        o.destroy()
    d.qfDiagnostic = ceed.QFunction(1, opt["diagnostic"])
    d.qfDiagnostic.add_input("u", 3, EVAL_INTERP)
    d.qfDiagnostic.add_input("du", 9, EVAL_GRAD)
    d.qfDiagnostic.add_input("qdata", qdatasize, EVAL_NONE)
    d.qfDiagnostic.add_output("diagnostic", 8, EVAL_NONE)
    d.qfDiagnostic.set_context(phys)
    d.opDiagnostic = ceed.Operator(d.qfDiagnostic)
    d.opDiagnostic.set_field("u", d.Erestrictu, d.basisDiagnostic, VECTOR_ACTIVE)
    d.opDiagnostic.set_field("du", d.Erestrictu, d.basisDiagnostic, VECTOR_ACTIVE)
    d.opDiagnostic.set_field("qdata", d.ErestrictqdDiagnostici, BASIS_COLLOCATED, d.qdataDiagnostic)
    d.opDiagnostic.set_field("diagnostic", d.ErestrictDiagnostic, BASIS_COLLOCATED, VECTOR_ACTIVE)
    return d.opDiagnostic


def setup_true_solution(ceed, mesh, data, P):
    """MMS true solution at the mesh nodes (setuplibceed.c:592-643), multiplicity-corrected."""
    d = data
    basisxtrue = ceed.BasisTensorH1Lagrange(3, 3, 2, P, GAUSS_LOBATTO)
    qf = ceed.QFunction(1, "qfunctions/manufacturedTrue.h:MMSTrueSoln")
    qf.add_input("x", 3, EVAL_INTERP)
    qf.add_output("true_soln", 3, EVAL_NONE)
    op = ceed.Operator(qf)
    op.set_field("x", d.Erestrictx, basisxtrue, VECTOR_ACTIVE)
    op.set_field("true_soln", d.Erestrictu, BASIS_COLLOCATED, VECTOR_ACTIVE)
    xcoord = d.Erestrictx.create_vector()
    xcoord.set_array(mesh.coord_lvector(), libceed.MEM_HOST, libceed.COPY_VALUES)
    truesoln = d.Erestrictu.create_vector()
    op.apply(xcoord, truesoln)
    mult = d.Erestrictu.create_vector()
    mult.set_value(0.0)
    d.Erestrictu.get_multiplicity(mult)
    out = truesoln.to_numpy() / mult.to_numpy()
    for o in (op, qf, basisxtrue, xcoord, truesoln, mult):
        o.destroy()
    return out


def setup_level(ceed, mesh, problem, degrees, level, phys, data, qextra=0, node_perm=None, multigrid=True,
                qf_locators=None):
    """SetupLibceedLevel (setuplibceed.c:748-863): data = list of CeedData, fine level last."""
    opt = problem_options(problem, qf_locators)
    fine = len(degrees) - 1
    P = degrees[level] + 1
    Q = degrees[fine] + 1 + qextra
    dim = ncompu = 3
    qdatasize = opt["qdatasize"]
    d, df = data[level], data[fine]
    if level != fine:
        d.Erestrictu = create_restriction(ceed, mesh, P, ncompu, node_perm if level == fine else None)
        d.basisu = ceed.BasisTensorH1Lagrange(dim, ncompu, P, Q, opt["qmode"])
    if level != 0:
        d.basisCtoF = ceed.BasisTensorH1Lagrange(dim, ncompu, degrees[level - 1] + 1, P, GAUSS_LOBATTO)
    Ulocsz = ncompu * mesh.num_nodes(degrees[level])
    d.xceed = ceed.Vector(Ulocsz)
    d.yceed = ceed.Vector(Ulocsz)
    # -- Jacobian evaluator (:818-839)
    d.qfJacob = ceed.QFunction(1, opt["jacob"])
    d.qfJacob.add_input("deltadu", ncompu * dim, EVAL_GRAD)
    d.qfJacob.add_input("qdata", qdatasize, EVAL_NONE)
    if opt["nonlinear"]:
        d.qfJacob.add_input("gradu", ncompu * dim, EVAL_NONE)
    d.qfJacob.add_output("deltadv", ncompu * dim, EVAL_GRAD)
    # the reference passes sizeof(phys) == sizeof(pointer) here (:826); tolerated by the backend for its built-in
    # bodies.  A user Jacobian (qf_locators) is compiled at run time and given exactly ctxsize bytes: pass the struct.
    d.qfJacob.set_context(phys, size=None if qf_locators and "jacob" in qf_locators else 8)
    d.opJacob = ceed.Operator(d.qfJacob)
    d.opJacob.set_field("deltadu", d.Erestrictu, d.basisu, VECTOR_ACTIVE)
    d.opJacob.set_field("qdata", df.Erestrictqdi, BASIS_COLLOCATED, df.qdata)
    d.opJacob.set_field("deltadv", d.Erestrictu, d.basisu, VECTOR_ACTIVE)
    if opt["nonlinear"]:
        d.opJacob.set_field("gradu", df.ErestrictGradui, BASIS_COLLOCATED, df.gradu)
    # -- restriction and prolongation (:847-863)
    if level != 0 and multigrid:
        qfRestrict = ceed.QFunctionIdentity(ncompu, EVAL_NONE, EVAL_INTERP)
        qfProlong = ceed.QFunctionIdentity(ncompu, EVAL_INTERP, EVAL_NONE)
        d.opRestrict = ceed.Operator(qfRestrict)
        d.opRestrict.set_field("input", d.Erestrictu, BASIS_COLLOCATED, VECTOR_ACTIVE)
        d.opRestrict.set_field("output", data[level - 1].Erestrictu, d.basisCtoF, VECTOR_ACTIVE)
        d.opProlong = ceed.Operator(qfProlong)
        d.opProlong.set_field("input", data[level - 1].Erestrictu, d.basisCtoF, VECTOR_ACTIVE)
        d.opProlong.set_field("output", d.Erestrictu, BASIS_COLLOCATED, VECTOR_ACTIVE)
        d.keep += [qfRestrict, qfProlong]
    return d


def setup_all(ceed, mesh, problem, degree, nu=0.3, E=1.0, qextra=0, multigrid="logarithmic", node_perm=None,
              qf_locators=None):
    """The reference's set-up sequence (elasticity.c:255-281): fine level first, then every level
    coarse to fine.  Returns (degrees, [CeedData per level], phys).  qf_locators: {"apply": ..., "jacob": ...}
    overriding the problem's residual / Jacobian QFunction locators (problem_options); energy and diagnostic
    operators keep the problem's own."""
    problem_options(problem, qf_locators)  # reject bad keys before any device work
    degrees = level_degrees(degree, multigrid)
    phys = Physics(nu, E)
    data = [CeedData() for _ in degrees]
    setup_fine_level(ceed, mesh, problem, degree, phys, data[-1], qextra, node_perm, qf_locators)
    for level in range(len(degrees)):
        setup_level(ceed, mesh, problem, degrees, level, phys, data, qextra, node_perm, multigrid != "none",
                    qf_locators)
    return degrees, data, phys
