"""A conforming hex mesh whose elements are listed under random cube rotations (helpers.reoriented) is the same
discretisation as the original: HexMesh numbers the degree-p nodes topologically, so node ids, node count,
coordinates and Dirichlet masks agree, and the oracle operators agree to rounding.  The GPU tests use such meshes
to run the kernels with neighbours whose local axes differ."""
import numpy as np
import pytest

from ceedpetscsolid_b200.exodus import HexMesh, tube_mesh
from ceedpetscsolid_b200.mesh import BoxMesh, smooth_displacement
from helpers import OracleProblem, cube_rotations, reoriented
from oracle import oracle


def meshes():
    box = BoxMesh(n=(3, 2, 2), perturb=0.1, seed=1)
    return {"tube": tube_mesh(2, 8, 2), "sector": tube_mesh(2, 3, 2, angle=np.pi / 2),
            "box": HexMesh(box.vertices.reshape(-1, 3), box.offsets(1) // 3)}


def test_rotations_keep_every_element_positively_oriented():
    assert len(set(map(repr, cube_rotations()))) == 24
    a = tube_mesh(1, 24, 4)
    b = reoriented(a, seed=3)
    d = b.vertices[b.connect]
    # trilinear Jacobian at vertex 0 of every element: (v1 - v0) x (v2 - v0) . (v4 - v0) > 0
    vol = np.einsum("ed,ed->e", np.cross(d[:, 1] - d[:, 0], d[:, 2] - d[:, 0]), d[:, 4] - d[:, 0])
    assert (vol > 0).all()
    # the elements really are listed differently: vertex 0 is a different corner for most of them
    assert (b.connect[:, 0] != a.connect[:, 0]).mean() > 0.5


@pytest.mark.parametrize("name", ["tube", "sector", "box"])
@pytest.mark.parametrize("p", [1, 2, 3, 4])
def test_reoriented_mesh_has_the_same_nodes(name, p):
    a = meshes()[name]
    b = reoriented(a, seed=p)
    assert not np.array_equal(a.connect, b.connect)
    assert b.num_nodes(p) == a.num_nodes(p)
    ia, ib = a.offsets(p) // 3, b.offsets(p) // 3
    assert np.array_equal(np.sort(ia, axis=1), np.sort(ib, axis=1))     # each element holds the same node ids
    # a shared node's coordinates come from whichever element lists it last, so a rotated listing may round them
    # differently in the last bit
    xa = a.node_coords(p)
    np.testing.assert_allclose(b.node_coords(p), xa, rtol=0, atol=4 * np.finfo(float).eps * np.abs(xa).max())
    assert np.array_equal(b.boundary_mask(p), a.boundary_mask(p))
    for ss in a.sidesets:
        assert np.array_equal(b.boundary_mask(p, [ss]), a.boundary_mask(p, [ss])), ss


def max_rel(got, ref):
    return np.abs(got - ref).max() / np.abs(ref).max()


@pytest.mark.parametrize("problem", ["linElas", "hyperSS", "hyperFS"])
@pytest.mark.parametrize("name,p", [("tube", 2), ("box", 3), ("sector", 4)])
def test_oracle_operators_agree_on_the_reoriented_mesh(problem, name, p):
    a = meshes()[name]
    b = reoriented(a, seed=7)
    oa, ob = OracleProblem(problem, None, p, mesh=a), OracleProblem(problem, None, p, mesh=b)
    u = smooth_displacement(a.node_coords(p), 0.05).reshape(-1)
    assert max_rel(ob.residual_fine(u), oa.residual_fine(u)) <= 1e-13
    x = np.random.default_rng(p).standard_normal(oa.lsize)
    assert max_rel(ob.jacobian(x), oa.jacobian(x)) <= 1e-13
    assert max_rel(ob.diagonal(), oa.diagonal()) <= 1e-13
    xc = np.random.default_rng(p + 1).standard_normal(a.lsize(p - 1))
    pa = oracle.transfer(False, a.nelem, p, p + 1, a.offsets(p - 1), a.offsets(p), xc, a.lsize(p))
    pb = oracle.transfer(False, b.nelem, p, p + 1, b.offsets(p - 1), b.offsets(p), xc, b.lsize(p))
    assert max_rel(pb, pa) <= 1e-13
