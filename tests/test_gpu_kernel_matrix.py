"""GPU: every volume-kernel instance the operators can select, every quadrature rule the API accepts, the element metrics and
the linear functionals, each against the plain FP64 reference of tests/fp64_ref.py.

The instance tables below restate find_instance / find_tpe_instance / find_pair_instance / find_affine_instance of
csrc/operators.cu, and expect() restates select_volume_kernel. Every case runs under every knob that routes it to a
different kernel family and asserts the family it expects, so a change of the selection code cannot silently move a case off
the kernel it exists to cover. Operator tolerance: 1e-12 relative in l2, as in test_gpu_parity.py."""
import numpy as np
import pytest
import torch

import cuddhelmholtz_b200 as cb
from conftest import load_mesh_file
from fp64_ref import GL, GLL, Faces, Space, interior_edges
from gpu_util import dev, host, max_ctas, rel, warped_mesh
from oracle import ops as O
from oracle import setup_np as S

pytestmark = pytest.mark.gpu
TOL = 1e-12

_DEFAULT = [(2, 3), (3, 4), (4, 5), (5, 6), (6, 7), (7, 8), (8, 9), (9, 10)]  # nq = nb + 1
_PLUS2 = [(3, 5), (4, 6), (5, 7), (6, 8), (7, 9), (8, 10)]                     # nq = nb + 2
_WEIGHTED = [(2, 5), (3, 6), (4, 8), (5, 9), (6, 11), (7, 12), (8, 14), (9, 15)]  # nq = 1 + 3nb/2 + 1
LANE = {"S": _DEFAULT + _PLUS2, "M": _DEFAULT + _PLUS2 + _WEIGHTED}                 # find_instance
TPE = {"S": [(2, 3), (3, 4), (4, 5), (5, 6), (3, 5), (4, 6), (5, 7)],             # find_tpe_instance
       "M": [(2, 3), (3, 4), (4, 5), (5, 6), (3, 5), (4, 6), (5, 7), (2, 5), (3, 6), (4, 8), (5, 9)]}
PAIR = {"S": [(6, 7), (7, 8), (8, 9), (9, 10)],                                    # find_pair_instance (S, nb 9: affine only)
        "M": [(6, 7), (7, 8), (8, 9), (9, 10), (6, 11), (7, 12), (8, 14), (9, 15)]}
AFFINE_TPE = [(4, 5), (5, 6)]                                                      # find_affine_instance
NO_INSTANCE = {"S": [(2, 2), (5, 8), (9, 11)], "M": [(3, 3), (6, 9), (9, 16)]}    # generic kernel
KNOBS = {"default": {}, "TPE0": {"CUDDH_B200_TPE": "0"}, "PAIR0": {"CUDDH_B200_PAIR": "0"},
         "GENERIC": {"CUDDH_B200_FORCE_GENERIC": "1"}, "AFFINE0": {"CUDDH_B200_AFFINE": "0"}, "FUSED0": {"CUDDH_B200_FUSED": "0"}}
ALL_KNOBS = sorted({k for v in KNOBS.values() for k in v} | {"CUDDH_B200_RING1", "CUDDH_B200_RING4", "CUDDH_B200_TPE_PX",
                                                             "CUDDH_B200_TPE_PY", "CUDDH_B200_PX", "CUDDH_B200_PY"})


def expect(op, nb, nq, knob, gauss=True, affine_mesh=True):
    """(kernel_kind, is_affine, family name) that select_volume_kernel picks; the affine formulation needs a stiffness
    operator, a Gauss-Legendre rule and a mesh of parallelograms"""
    if knob == "GENERIC" or (nb, nq) not in LANE[op]:
        return 0, False, "generic"
    aff = op == "S" and gauss and knob != "AFFINE0" and affine_mesh
    if knob != "TPE0" and (nb, nq) in TPE[op]:
        return 1, aff and (nb, nq) in AFFINE_TPE, "tpe"
    if knob != "PAIR0" and (nb, nq) in PAIR[op] and not (op == "S" and nb == 9 and not aff):
        return 3, aff, "pair"
    return 0, False, "lane"


def _cases():
    out = []
    for op in ("S", "M"):
        for nb, nq in LANE[op]:
            knobs = ["default", "GENERIC"]
            knobs += ["TPE0"] if (nb, nq) in TPE[op] else []
            knobs += ["PAIR0"] if (nb, nq) in PAIR[op] else []
            knobs += ["AFFINE0"] if op == "S" and ((nb, nq) in AFFINE_TPE or (nb, nq) in PAIR[op]) else []
            out += [(op, nb, nq, k) for k in knobs]
        out += [(op, nb, nq, "default") for nb, nq in NO_INSTANCE[op]]
    return out


CASES = _cases()


def _case_id(c):
    op, nb, nq, knob = c
    return "%s-nb%d-nq%d-%s-%s" % (op, nb, nq, knob, expect(op, nb, nq, knob)[2])  # family on an affine mesh


def _set_knobs(monkeypatch, knob):
    for k in ALL_KNOBS:
        monkeypatch.delenv(k, raising=False)
    for k, v in KNOBS[knob].items():
        monkeypatch.setenv(k, v)


# meshes and their persistent-CTA cap (0: none). rect_aniso: affine, non-square elements, ragged patch tiling and partial
# warp passes; warp12: every element its own metric; unstr: the golden unstructured mesh; warp24 under max_ctas(2): several
# patches per persistent CTA, so the metric rings wrap across patches
MESHES = {"rect_aniso": 0, "warp12": 0, "unstr": 0, "warp24": 2}
_cache = {}


def _mesh(tag):
    if tag not in _cache:
        if tag == "rect_aniso":
            _cache[tag] = cb.Mesh2D.uniform_rect(13, -1.0, 2.0, 7, 0.0, 1.0)
        elif tag.startswith("warp"):
            _cache[tag] = cb.Mesh2D.from_vertices(*warped_mesh(int(tag[4:])))
        else:
            _cache[tag] = cb.Mesh2D.from_vertices(*load_mesh_file())
    return _cache[tag]


def _affine(mesh):
    C = mesh.vertices()[mesh.elements()]
    return bool(np.abs(C[:, 0] - C[:, 1] + C[:, 2] - C[:, 3]).max() <= 1e-14 * np.abs(C).max())


def _space(tag, nb):
    key = (tag, nb)
    if key not in _cache:
        fem = cb.H1Space(_mesh(tag), cb.Basis(nb))
        _cache[key] = (fem, Space(fem))
    return _cache[key]


def _vec(n, seed):
    return np.random.default_rng(seed).uniform(-1.0, 1.0, n)


def _coef(xy):
    return 1.0 + 0.5 * np.sin(np.pi * xy[:, 0]) * np.cos(np.pi * xy[:, 1])


def _check_operator(P, ref, n, name):
    """action(x, y) over garbage, action(-0.75, x, y) on a non-zero y, bitwise repeatability; ref(x, c, y0) -> y0 + c A x"""
    x = _vec(n, 11)
    dx = dev(x)
    y = torch.full((n,), 7.0, dtype=torch.float64, device="cuda")
    P.action(dx, y)
    e = rel(host(y), ref(x, 1.0, None))
    assert e < TOL, (name, "overwrite", e)
    y0 = _vec(n, 12)
    dy = dev(y0)
    P.action(-0.75, dx, dy)
    e = rel(host(dy), ref(x, -0.75, y0))
    assert e < TOL, (name, "accumulate", e)
    y2 = torch.full((n,), -3.0, dtype=torch.float64, device="cuda")
    P.action(dx, y2)
    assert torch.equal(y, y2), (name, "not bitwise repeatable")


@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_volume_kernel_matrix(case, monkeypatch):
    op, nb, nq, knob = case
    _set_knobs(monkeypatch, knob)
    for tag, cap in MESHES.items():
        fem, sp = _space(tag, nb)
        n = sp.ndof
        kind, aff, _ = expect(op, nb, nq, knob, affine_mesh=_affine(_mesh(tag)))
        with max_ctas(cap):
            if op == "S":
                P = cb.StiffnessMatrix(fem, cb.QuadratureRule(nq, cb.GaussLegendre))
                variants = [(P, lambda x, c, y0: sp.stiffness(x, nq, GL, c, y0), "S")]
            else:
                a = _coef(sp.xy)
                da = dev(a)
                variants = [(cb.MassMatrix(fem, n_quad=nq), lambda x, c, y0: sp.mass(x, nq, None, c, y0), "M"),
                            (cb.MassMatrix(da, fem, n_quad=nq), lambda x, c, y0: sp.mass(x, nq, a, c, y0), "Mw")]
            for P, ref, name in variants:
                assert P.kernel_kind() == kind, (tag, name, P.kernel_kind(), kind)
                assert P.is_affine() == aff, (tag, name, P.is_affine())
                _check_operator(P, ref, n, (tag, name))


# ---- the Helmholtz composite under each knob that takes it off the fused default ----------------------------------------
def _helm_kind(nb, knob, affine_mesh):
    ks, sa, _ = expect("S", nb, nb + 1, knob, affine_mesh=affine_mesh)
    km, _, _ = expect("M", nb, 1 + 3 * nb // 2 + 1, knob)
    fused = knob != "FUSED0" and ks == km and ((ks == 1 and nb <= 5 and (not sa or nb >= 4)) or (ks == 3 and sa))
    return 2 if fused else ks


_oracle_cache = {}


def _oracle_space(tag, nb):
    if (tag, nb) not in _oracle_cache:
        if tag == "rect_aniso":
            om = S.uniform_rect(13, -1.0, 2.0, 7, 0.0, 1.0)
        elif tag.startswith("warp"):
            om = S.mesh_from_vertices(*warped_mesh(int(tag[4:])))
        else:
            om = S.mesh_from_vertices(*load_mesh_file())
        ofem = O.H1(om, nb)
        _oracle_cache[(tag, nb)] = (ofem, O.FaceSpace(ofem, om.boundary_edges))
    return _oracle_cache[(tag, nb)]


@pytest.mark.parametrize("knob", ["FUSED0", "TPE0", "PAIR0", "GENERIC"])
@pytest.mark.parametrize("nb", [4, 5, 8])
def test_helmholtz_composite_fallbacks(nb, knob, monkeypatch):
    _set_knobs(monkeypatch, knob)
    omega = 10.0
    for tag in ("rect_aniso", "warp12"):
        fem, sp = _space(tag, nb)
        ofem, ofs = _oracle_space(tag, nb)
        assert np.array_equal(fem.global_indices().ravel(), ofem.I)
        fs = cb.FaceSpace(fem, _mesh(tag).boundary_edges())
        n = sp.ndof
        c = _coef(sp.xy)
        a2, af = c * c, c[ofs.proj]
        A = cb.Helmholtz(omega, dev(a2), dev(af), fem, fs)
        assert A.kernel_kind() == _helm_kind(nb, knob, _affine(_mesh(tag))), (tag, A.kernel_kind())
        x = _vec(2 * n, 21)
        y = torch.full((2 * n,), 5.0, dtype=torch.float64, device="cuda")
        A.action(dev(x), y)
        want = O.Helmholtz(omega, a2, af, ofem, ofs).action(x)
        got = host(y)
        # each block row on its own (a wrong-field read would otherwise average out in the joint norm)
        assert rel(got[:n], want[:n]) < TOL and rel(got[n:], want[n:]) < TOL, (tag, rel(got[:n], want[:n]), rel(got[n:], want[n:]))
        y2 = torch.empty_like(y)
        A.action(dev(x), y2)
        assert torch.equal(y, y2)


# ---- quadrature rules the API accepts --------------------------------------------------------------------------------------
QUAD_MESHES = ["rect_aniso", "unstr"]


@pytest.mark.parametrize("nb", [2, 4, 5, 8, 9])
def test_stiffness_quadrature_rules(nb, monkeypatch):
    _set_knobs(monkeypatch, "default")
    rules = [(nb + 1, GLL), (nb, GLL), (max(nb - 1, 1), GL), (1, GL), (24, GL)]
    for tag in QUAD_MESHES:
        fem, sp = _space(tag, nb)
        for nq, kind in rules:
            P = cb.StiffnessMatrix(fem, cb.QuadratureRule(nq, cb.GaussLobatto if kind == GLL else cb.GaussLegendre))
            k, aff, _ = expect("S", nb, nq, "default", gauss=kind == GL, affine_mesh=_affine(_mesh(tag)))
            assert P.kernel_kind() == k, (tag, nq, kind, P.kernel_kind())
            # a Gauss-Lobatto rule never takes the affine formulation, even on an affine mesh
            assert P.is_affine() == aff, (tag, nq, kind)
            if kind == GLL and tag == "rect_aniso":
                assert not P.is_affine()
            _check_operator(P, lambda x, c, y0: sp.stiffness(x, nq, kind, c, y0), sp.ndof, (tag, nq, kind))
        with pytest.raises(cb.CuddhError):
            cb.StiffnessMatrix(fem, cb.QuadratureRule(25, cb.GaussLegendre))


@pytest.mark.parametrize("nb", [2, 4, 5, 8, 9])
def test_mass_quadrature_rules(nb, monkeypatch):
    _set_knobs(monkeypatch, "default")
    rules = sorted({1, max(nb - 1, 1), nb + 1, nb + 2, 1 + 3 * nb // 2 + 1, 32})
    for tag in QUAD_MESHES:
        fem, sp = _space(tag, nb)
        a = _coef(sp.xy)
        da = dev(a)
        for nq in rules:
            for P, coef in [(cb.MassMatrix(fem, n_quad=nq), None), (cb.MassMatrix(da, fem, n_quad=nq), a)]:
                assert P.kernel_kind() == expect("M", nb, nq, "default")[0], (tag, nq)
                _check_operator(P, lambda x, c, y0: sp.mass(x, nq, coef, c, y0), sp.ndof, (tag, nq, coef is not None))
        with pytest.raises(cb.CuddhError):
            cb.MassMatrix(fem, n_quad=33)
        with pytest.raises(cb.CuddhError):
            cb.MassMatrix(da, fem, n_quad=33)


def _face_spaces(tag, nb):
    fem, sp = _space(tag, nb)
    mesh = _mesh(tag)
    return [("boundary", cb.FaceSpace(fem, mesh.boundary_edges())), ("interior", cb.FaceSpace(fem, interior_edges(mesh)))]


@pytest.mark.parametrize("nb", [2, 4, 5, 8])
def test_face_mass_quadrature_rules(nb):
    rules = sorted({1, nb, nb + 1, 1 + 3 * nb // 2 + 1, 64})
    for tag in QUAD_MESHES:
        fem, sp = _space(tag, nb)
        for fname, fs in _face_spaces(tag, nb):
            fc = Faces(sp, fs)
            nf = fs.size()
            af = _coef(sp.xy[fc.proj])
            daf = dev(af)
            u = _vec(sp.ndof, 31)
            du = dev(u)
            for nq in rules:
                for H, coef in [(cb.FaceMassMatrix(fs, n_quad=nq), None), (cb.FaceMassMatrix(daf, fs, n_quad=nq), af)]:
                    name = (tag, fname, nq, coef is not None)
                    _check_operator(H, lambda x, c, y0: fc.mass(x, nq, coef, c, y0), nf, name)
                    # fused restrict + action + prolong on H1 vectors
                    y0 = _vec(sp.ndof, 32)
                    dy = dev(y0)
                    H.action_h1(-1.5, du, dy)
                    want = fc.prolong(fc.mass(fc.restrict(u), nq, coef, -1.5), y0)
                    assert rel(host(dy), want) < TOL, name
            with pytest.raises(cb.CuddhError):
                cb.FaceMassMatrix(fs, n_quad=65)
            with pytest.raises(cb.CuddhError):
                cb.FaceMassMatrix(daf, fs, n_quad=65)


def test_empty_face_space_is_a_no_op():
    fem, sp = _space("unstr", 4)
    fs = cb.FaceSpace(fem, np.zeros(0, np.int32))
    assert fs.size() == 0 and fs.subspace_indices().shape == (0, 4)
    e = torch.empty(0, dtype=torch.float64, device="cuda")
    u = dev(_vec(sp.ndof, 41))
    y = dev(_vec(sp.ndof, 42))
    y_before = y.clone()
    fs.restrict(u, e)
    fs.prolong(e, y)
    fs.orth(y)
    for nq in (0, 1, 64):
        for H in (cb.FaceMassMatrix(fs, n_quad=nq), cb.FaceMassMatrix(e, fs, n_quad=nq)):
            H.action(e, e)
            H.action(2.0, e, e)
            H.action_h1(-1.5, u, y)
    cb.DiagInvFaceMassMatrix(fs).action(e, e)
    cb.FaceLinearFunctional(fs).action(lambda x, y_: x + y_, e)
    cb.FaceLinearFunctional(fs, cb.QuadratureRule(5, cb.GaussLegendre)).action(0.5, lambda x, y_: x + y_, e)
    torch.cuda.synchronize()
    assert torch.equal(y, y_before)


# ---- element metrics and linear functionals ----------------------------------------------------------------------------------
def _f(x, y):
    """neither symmetric under x -> -x nor under y -> -y: a reversed face or a transposed element shows"""
    return x + 2.0 * y ** 3 + x * y


def _g(x, y):
    return 1.0 + 0.5 * x * x - 0.25 * y


@pytest.mark.parametrize("tag", ["rect_aniso", "warp12", "unstr"])
@pytest.mark.parametrize("nb", [2, 4, 5, 8])
def test_metrics_and_linear_functionals(tag, nb):
    fem, sp = _space(tag, nb)
    n = sp.ndof
    for nq in sorted({1, nb, nb + 2, 16}):
        xq, _ = S.gauss_legendre(nq)
        for which in ("jacobians", "measures", "physical_coordinates"):
            got = host(fem.element_metrics(xq, which))
            want = sp.element_metrics(xq, which)
            assert got.shape == want.shape and rel(got, want) < 1e-13, (which, nq)
        rules = [(None, None), (cb.QuadratureRule(nq, cb.GaussLegendre), GL)]
        if nq >= 2:
            rules.append((cb.QuadratureRule(nq, cb.GaussLobatto), GLL))
        for quad, kind in rules:
            q = None if quad is None else nq
            name = (nq, kind)
            lf = cb.LinearFunctional(fem, quad)
            F = torch.full((n,), 3.0, dtype=torch.float64, device="cuda")  # action(f, F) overwrites
            lf.action(_f, F)
            want = sp.linear_functional(_f, q, kind)
            assert rel(host(F), want) < TOL, name
            lf.action(-0.5, _g, F)
            assert rel(host(F), sp.linear_functional(_g, q, kind, -0.5, want)) < TOL, name
            for fname, fs in _face_spaces(tag, nb):
                fc = Faces(sp, fs)
                fl = cb.FaceLinearFunctional(fs, quad)
                G = torch.full((fs.size(),), -2.0, dtype=torch.float64, device="cuda")
                fl.action(_f, G)
                want = fc.linear_functional(_f, q, kind)
                assert rel(host(G), want) < TOL, (fname,) + name
                fl.action(-0.5, _g, G)
                assert rel(host(G), fc.linear_functional(_g, q, kind, -0.5, want)) < TOL, (fname,) + name
