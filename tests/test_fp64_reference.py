"""CPU: the plain NumPy FP64 reference of tests/fp64_ref.py against the oracle (oracle/ops.py over oracle/oracle.c) on the
default rules, and against identities it must satisfy exactly. The GPU kernel tests (test_gpu_kernel_matrix.py) compare
with this reference, so a wrong reference would hide a wrong kernel."""
import numpy as np
import pytest

import cuddhelmholtz_b200 as cb
from conftest import load_mesh_file
from fp64_ref import GL, GLL, Faces, Space, interior_edges
from oracle import ops as O
from oracle import setup_np as S

TOL = 1e-13


def _meshes(kind):
    if kind == "rect":
        args = (6, -1.0, 2.0, 5, 0.0, 1.0)
        return S.uniform_rect(*args), cb.Mesh2D.uniform_rect(*args)
    xy, el = load_mesh_file()
    return S.mesh_from_vertices(xy, el), cb.Mesh2D.from_vertices(xy, el)


def _rel(a, b):
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def _spaces(kind, nb):
    om, pm = _meshes(kind)
    ofem = O.H1(om, nb)
    pfem = cb.H1Space(pm, cb.Basis(nb))
    assert np.array_equal(pfem.global_indices().ravel(), ofem.I)
    ofs = O.FaceSpace(ofem, om.boundary_edges)
    pfs = cb.FaceSpace(pfem, pm.boundary_edges())
    sp = Space(pfem)
    return om, pm, ofem, ofs, sp, Faces(sp, pfs)


def _area(pm):
    C = pm.vertices()[pm.elements()]
    x, y = C[..., 0], C[..., 1]
    return float(0.5 * np.sum(x * np.roll(y, -1, 1) - np.roll(x, -1, 1) * y))


@pytest.mark.parametrize("kind", ["rect", "unstr"])
@pytest.mark.parametrize("nb", [2, 4, 5, 8])
def test_reference_matches_oracle_on_default_rules(kind, nb):
    om, pm, ofem, ofs, sp, fc = _spaces(kind, nb)
    rng = np.random.default_rng(nb)
    u = rng.uniform(-1.0, 1.0, ofem.ndof)
    y0 = rng.uniform(-1.0, 1.0, ofem.ndof)
    a2 = 1.0 + 0.5 * np.sin(np.pi * ofem.xy[:, 0]) * np.cos(np.pi * ofem.xy[:, 1])
    assert _rel(sp.stiffness(u), O.StiffnessMatrix(ofem).action(u)) < TOL
    assert _rel(sp.stiffness(u, c=-0.75, y0=y0), O.StiffnessMatrix(ofem).action(u, y0.copy(), -0.75)) < TOL
    assert _rel(sp.stiffness(u, nq=nb + 2), O.StiffnessMatrix(ofem, nb + 2).action(u)) < TOL
    assert _rel(sp.mass(u), O.MassMatrix(ofem).action(u)) < TOL
    assert _rel(sp.mass(u, coef=a2), O.MassMatrix(ofem, a2).action(u)) < TOL
    assert _rel(sp.mass(u, coef=a2, c=2.5, y0=y0), O.MassMatrix(ofem, a2).action(u, y0.copy(), 2.5)) < TOL
    uf = fc.restrict(u)
    af = a2[fc.proj]
    assert np.array_equal(fc.proj, ofs.proj) and np.array_equal(uf, ofs.restrict(u))
    assert _rel(fc.mass(uf), O.FaceMassMatrix(ofs).action(uf)) < TOL
    assert _rel(fc.mass(uf, coef=af), O.FaceMassMatrix(ofs, af).action(uf)) < TOL
    from test_oracle_golden import _lf
    f = lambda x, y: x + 2.0 * y ** 3 + x * y
    assert _rel(sp.linear_functional(f, nb + 2), _lf(ofem, nb + 2, f)) < TOL


@pytest.mark.parametrize("kind", ["rect", "unstr"])
@pytest.mark.parametrize("nb", [2, 3, 5, 9])
def test_reference_identities(kind, nb):
    om, pm, ofem, ofs, sp, fc = _spaces(kind, nb)
    one = np.ones(sp.ndof)
    u = np.random.default_rng(3).uniform(-1.0, 1.0, sp.ndof)
    for nq, k in [(nb + 1, GL), (nb + 2, GL), (nb + 1, GLL), (nb, GLL)]:
        assert np.abs(sp.stiffness(one, nq, k)).max() <= 1e-13 * np.abs(sp.stiffness(u, nq, k)).max()
    area = _area(pm)
    for nq in (nb + 1, nb + 2, 1 + 3 * nb // 2 + 1):
        M1 = sp.mass(one, nq)
        assert abs(M1.sum() - area) <= 1e-13 * area
        assert abs(sp.mass(one, nq, coef=one).sum() - area) <= 1e-13 * area
    M1 = sp.mass(one)
    for nq in (nb + 1, nb + 2):
        assert _rel(sp.linear_functional(lambda x, y: np.ones_like(x), nq), M1) < TOL
    # faces: boundary FaceSpace and the interior edges
    for faces in (pm.boundary_edges(), interior_edges(pm)):
        f = Faces(sp, cb.FaceSpace(sp.fem, faces))
        V = pm.vertices()
        E = pm.edges()[faces]
        length = float(np.linalg.norm(V[E[:, 1]] - V[E[:, 0]], axis=1).sum())
        assert abs(2.0 * f.meas.sum() - length) <= 1e-13 * length
        for nq in (None, nb + 1):
            assert abs(f.linear_functional(lambda x, y: np.ones_like(x), nq).sum() - length) <= 1e-13 * length
        lin = lambda x, y: 0.25 + 2.0 * x - 3.0 * y
        pos = sp.xy[f.proj]
        assert _rel(f.linear_functional(lin, nb + 1), f.mass(lin(pos[:, 0], pos[:, 1]))) < TOL


@pytest.mark.parametrize("kind", ["rect", "unstr"])
def test_reference_metrics_match_oracle(kind):
    om, pm, ofem, ofs, sp, fc = _spaces(kind, 4)
    for nq in (1, 4, 7):
        x, _ = S.gauss_legendre(nq)
        nel = pm.n_elem()
        # the oracle's element arrays are column-major (2, 2, nq, nq, nel) / (nq, nq, nel) / (2, nq, nq, nel)
        assert _rel(sp.element_metrics(x, "jacobians").ravel(), ofem.jacobians(x).reshape(nel, nq, nq, 2, 2).ravel()) < TOL
        assert _rel(sp.element_metrics(x, "measures").ravel(), ofem.measures(x)) < TOL
        assert _rel(sp.element_metrics(x, "physical_coordinates").ravel(), ofem.coordinates(x)) < TOL
