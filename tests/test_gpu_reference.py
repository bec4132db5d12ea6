"""GPU: the CUDA path against the UNMODIFIED reference's own CUDA kernels, run through oracle/_ref/ref_driver when that
driver has been built (oracle/Makefile, from the reference's sources, which are not part of this repository): the strongest
parity pin.

Without the driver, the operator and GMRES commands are answered by the oracle instead (oracle/ops.py over oracle/oracle.c,
the CPU restatement of the reference's kernels: tests/test_oracle_golden.py pins its 1-D tables and index maps bit for bit to
the reference's own host objects and its operators to the reference tests' analytic KATs), on seeded inputs made here. The
assertions and tolerances are the same either way. The commands the oracle does not restate (element metrics / linear
functionals, DDH constructor tables) skip without the driver."""
import os
import subprocess
import tempfile

import numpy as np
import pytest
import torch

import cuddhelmholtz_b200 as cb
from conftest import MESH_FILE, REF_DRIVER, load_mesh_file
from gpu_util import dev, host, max_ctas, rel, warped_mesh, write_mesh_file
from oracle.rdmp import read_rdmp

pytestmark = pytest.mark.gpu


def ref(*args, timeout=600):
    if not os.path.exists(REF_DRIVER):
        return oracle_ref(*args)
    with tempfile.NamedTemporaryFile(suffix=".bin") as f:
        subprocess.check_call([REF_DRIVER, *[str(a) for a in args], f.name], timeout=timeout)
        return read_rdmp(f.name)


def _coef(xy):
    return 1.0 + 0.5 * np.sin(np.pi * xy[:, 0]) * np.cos(np.pi * xy[:, 1])


def _oracle_space(spec, nb):
    """oracle H1 space and boundary face space of a ref_driver mesh spec (rect:<nx> or file:<path>)"""
    from oracle import ops as O
    from oracle import setup_np as S
    if spec.startswith("rect:"):
        nx = int(spec[5:])  # closed form: pinned bit for bit to the first-touch numbering by tests/test_oracle_golden.py
        c = S.uniform_rect_closed_form(nx, -1.0, 1.0, nx, -1.0, 1.0, S.Basis(nb))
        fem = O.H1.from_arrays(nb, c["I"], c["xy"], c["corners"])
        return fem, O.FaceSpace.from_arrays(fem, c["face_I"], c["face_proj"], c["face_meas"])
    mesh = S.mesh_from_vertices(*load_mesh_file(spec[5:]))
    fem = O.H1(mesh, nb)
    return fem, O.FaceSpace(fem, mesh.boundary_edges)


def oracle_ref(cmd, *args):
    """the ref_driver commands ops / ops_lite / helm_gmres (oracle/ref_driver.cu), same keys, computed by the oracle"""
    from oracle import ops as O
    if cmd not in ("ops", "ops_lite", "helm_gmres"):
        pytest.skip("ref_driver %s needs the reference's build (oracle/_ref/ref_driver)" % cmd)
    spec, nb, omega = args[0], int(args[1]), float(args[2])
    fem, fs = _oracle_space(spec, nb)
    n, nf = fem.ndof, fs.fdof
    c = _coef(fem.xy)
    a2, af = c * c, c[fs.proj]
    r = {"ndof": np.array([n]), "fdof": np.array([nf]), "a2": a2, "af": af}
    if cmd == "helm_gmres":
        m, maxit, tol = int(args[3]), int(args[4]), float(args[5])
        s = omega * omega  # two point sources, mass-weighted into the first block
        X, Y = fem.xy[:, 0], fem.xy[:, 1]
        src = s / np.pi * np.exp(-s * ((X + 0.5) ** 2 + Y ** 2)) + s / np.pi * np.exp(-s * ((X - 0.5) ** 2 + (Y + 0.5) ** 2))
        b = np.concatenate([O.MassMatrix(fem).action(src), np.zeros(n)])
        U = np.zeros(2 * n)
        out = O.gmres(2 * n, U, O.Helmholtz(omega, a2, af, fem, fs).action, b, m, maxit, tol)
        r.update(b=b, U=U, success=np.array([int(out["success"])]), num_iter=np.array([out["num_iter"]]),
                 num_matvec=np.array([out["num_matvec"]]), res_norm=np.array(out["res_norm"]))
        return r
    rng = np.random.default_rng(int(args[3]))
    X = rng.uniform(-1.0, 1.0, 2 * n)
    r["helm_x"] = X
    r["helm_Ax"] = O.Helmholtz(omega, a2, af, fem, fs).action(X)
    S_, Mw = O.StiffnessMatrix(fem), O.MassMatrix(fem, a2)
    if cmd == "ops_lite":
        u, v = X[:n], X[n:]
        r["S_u"] = S_.action(u)
        r["S_acc"] = S_.action(v, r["S_u"].copy(), -0.75)
        r["Mw_u"] = Mw.action(u)
        r["Mw_acc"] = Mw.action(v, r["Mw_u"].copy(), 2.5)
        return r
    f_s, f_m = rng.uniform(-1.0, 1.0, n), rng.uniform(-1.0, 1.0, n)
    r.update(f_stiff=f_s, f_mass=f_m)
    r["S_default_f"] = S_.action(f_s)
    r["S_default_acc"] = S_.action(f_m, r["S_default_f"].copy(), -0.75)
    r["S_q2_f"] = O.StiffnessMatrix(fem, nb + 2).action(f_s)
    r["M_f"] = O.MassMatrix(fem).action(f_m)
    r["Mw_f"] = Mw.action(f_m)
    r["Mw_acc"] = Mw.action(f_s, r["Mw_f"].copy(), 2.5)
    r["Mi_f"] = O.DiagInvMassMatrix(fem).action(f_m)
    r["Miw_f"] = O.DiagInvMassMatrix(fem, a2).action(f_m)
    xf = fs.restrict(f_m)
    r["restrict_f"] = xf
    r["H_f"] = O.FaceMassMatrix(fs).action(xf)
    r["Hw_f"] = O.FaceMassMatrix(fs, af).action(xf)
    r["Hi_f"] = O.DiagInvFaceMassMatrix(fs).action(xf)
    r["prolong"] = fs.prolong(r["Hi_f"], f_s.copy())
    r["orth"] = fs.orth(r["prolong"].copy())
    return r


SPREAD_NOTE = ("north_star: +-1; the reference's own count is not reproducible on long solves - FP32 shared-memory atomicAdd in "
               "source/DDH.cpp:108 - observed 80..82 restarts over three runs at (nx, n_basis) = (8, 8), against a bitwise reproducible 80 here")


def restart_slack(ref_it):
    """+-1 restart for every solve that converges within 30 restarts (north_star); longer solves get the reference's own
    run-to-run spread (about 2.5 % of the count, see SPREAD_NOTE), never less than 1"""
    return 1 if ref_it <= 30 else max(1, int(round(0.025 * ref_it)))


def product_mesh(spec):
    if spec.startswith("rect:"):
        nx = int(spec[5:])
        return cb.Mesh2D.uniform_rect(nx, -1.0, 1.0, nx, -1.0, 1.0)
    xy, el = load_mesh_file()
    return cb.Mesh2D.from_vertices(xy, el)


@pytest.mark.parametrize("spec", ["rect:10", "file:" + MESH_FILE, "rect:64"])
@pytest.mark.parametrize("nb", [4, 5, 8, 9])
def test_operator_actions_match_reference_kernels(spec, nb):
    if spec == "rect:64" and nb not in (4, 5):
        pytest.skip("large case only for the headline orders")
    omega = 10.0
    r = ref("ops", spec, nb, omega, 12345)
    mesh = product_mesh(spec)
    fem = cb.H1Space(mesh, cb.Basis(nb))
    fs = cb.FaceSpace(fem, mesh.boundary_edges())
    n, nf = fem.size(), fs.size()
    assert n == r["ndof"][0] and nf == r["fdof"][0]
    f_s, f_m, a2, af = dev(r["f_stiff"]), dev(r["f_mass"]), dev(r["a2"]), dev(r["af"])
    y = torch.empty(n, dtype=torch.float64, device="cuda")
    tol = 1e-12

    S = cb.StiffnessMatrix(fem)
    S.action(f_s, y)
    assert rel(host(y), r["S_default_f"]) < tol
    S.action(-0.75, f_m, y)
    assert rel(host(y), r["S_default_acc"]) < tol
    cb.StiffnessMatrix(fem, cb.QuadratureRule(nb + 2, cb.GaussLegendre)).action(f_s, y)
    assert rel(host(y), r["S_q2_f"]) < tol

    cb.MassMatrix(fem).action(f_m, y)
    assert rel(host(y), r["M_f"]) < tol
    Mw = cb.MassMatrix(a2, fem)
    Mw.action(f_m, y)
    assert rel(host(y), r["Mw_f"]) < tol
    Mw.action(2.5, f_s, y)
    assert rel(host(y), r["Mw_acc"]) < tol
    cb.DiagInvMassMatrix(fem).action(f_m, y)
    assert rel(host(y), r["Mi_f"]) < tol
    cb.DiagInvMassMatrix(a2, fem).action(f_m, y)
    assert rel(host(y), r["Miw_f"]) < tol

    xf = torch.empty(nf, dtype=torch.float64, device="cuda")
    yf = torch.empty_like(xf)
    fs.restrict(f_m, xf)
    assert np.array_equal(host(xf), r["restrict_f"])
    cb.FaceMassMatrix(fs).action(xf, yf)
    assert rel(host(yf), r["H_f"]) < tol
    cb.FaceMassMatrix(af, fs).action(xf, yf)
    assert rel(host(yf), r["Hw_f"]) < tol
    cb.DiagInvFaceMassMatrix(fs).action(xf, yf)
    assert rel(host(yf), r["Hi_f"]) < tol
    y.copy_(f_s)
    fs.prolong(yf, y)
    assert rel(host(y), r["prolong"]) < 1e-15
    fs.orth(y)
    assert np.array_equal(host(y), r["orth"])

    A = cb.Helmholtz(omega, a2, af, fem, fs)
    Ax = torch.empty(2 * n, dtype=torch.float64, device="cuda")
    A.action(dev(r["helm_x"]), Ax)
    assert rel(host(Ax), r["helm_Ax"]) < tol


# Steady state of the persistent kernels (buffer rotation, metric-ring wrap across rows / phases / fields / patches, list
# prefetch, per-patch cluster barrier) against the reference's own kernels: every case gives each persistent CTA SEVERAL
# patches - by size (256^2: 512 patches on <= 296 CTAs; 1024^2: 8192) or by capping the CTA count - and the warped mesh gives
# every element its own metric block, so a stale ring slot or a wrong-patch read cannot hide.
# 4th entry: the stiffness formulation on uniform (all-affine) meshes - True = per-element metric constants (the default there),
# False = CUDDH_B200_AFFINE=0, the stored-metric ring kernels that every other mesh uses
STEADY = [("rect:64", 4, 8, True), ("rect:64", 5, 8, True), ("rect:64", 5, 2, False), ("rect:64", 4, 8, False),
          ("warp:200", 4, 16, False), ("warp:200", 5, 16, False), ("warp:256", 5, 0, False),
          ("rect:256", 4, 0, True), ("rect:256", 5, 0, True), ("rect:256", 5, 0, False), ("rect:256", 8, 0, False), ("warp:96", 8, 0, False),
          ("rect:1024", 5, 0, True)]


@pytest.mark.parametrize("spec,nb,cap,affine", STEADY)
def test_steady_state_matches_reference_kernels(spec, nb, cap, affine, tmp_path, monkeypatch):
    omega = 10.0
    if spec.startswith("rect:") and not affine:
        monkeypatch.setenv("CUDDH_B200_AFFINE", "0")
    if spec.startswith("warp:"):
        xy, el = warped_mesh(int(spec[5:]))
        path = str(tmp_path / "warped.txt")
        write_mesh_file(path, xy, el)
        rspec = "file:" + path
        mesh = cb.Mesh2D.from_vertices(xy, el)
    else:
        rspec = spec
        mesh = product_mesh(spec)
    r = ref("ops_lite", rspec, nb, omega, 4242, timeout=1500)
    fem = cb.H1Space(mesh, cb.Basis(nb))
    fs = cb.FaceSpace(fem, mesh.boundary_edges())
    n = fem.size()
    assert n == r["ndof"][0] and fs.size() == r["fdof"][0]
    a2, af, X = dev(r["a2"]), dev(r["af"]), dev(r["helm_x"])
    u, v = X[:n], X[n:]
    y = torch.empty(n, dtype=torch.float64, device="cuda")
    tol = 1e-12
    with max_ctas(cap):
        S = cb.StiffnessMatrix(fem)
        n_patch = fem.check_plan(1)["n_patches"] if nb <= 5 else 0
        if nb <= 5:
            assert S.kernel_kind() == 1 and S.is_affine() == affine
            ctas = cap if cap else 296
            assert n_patch >= 1.7 * ctas, (n_patch, ctas)  # several patches per persistent CTA
        S.action(u, y)
        assert rel(host(y), r["S_u"]) < tol
        S.action(-0.75, v, y)
        assert rel(host(y), r["S_acc"]) < tol
        Mw = cb.MassMatrix(a2, fem)
        Mw.action(u, y)
        assert rel(host(y), r["Mw_u"]) < tol
        Mw.action(2.5, v, y)
        assert rel(host(y), r["Mw_acc"]) < tol
        A = cb.Helmholtz(omega, a2, af, fem, fs)
        if nb <= 5:
            assert A.kernel_kind() == 2 and A.is_affine() == affine
        Ax = torch.empty(2 * n, dtype=torch.float64, device="cuda")
        A.action(X, Ax)
        assert rel(host(Ax), r["helm_Ax"]) < tol
        # each block row on its own as well (a wrong-field read would otherwise average out in the joint norm)
        assert rel(host(Ax[:n]), r["helm_Ax"][:n]) < tol and rel(host(Ax[n:]), r["helm_Ax"][n:]) < tol


@pytest.mark.parametrize("spec", ["rect:10", "file:" + MESH_FILE])
@pytest.mark.parametrize("nb,nq", [(4, 6), (5, 9), (8, 10)])
def test_metrics_and_linear_functionals_match_reference(spec, nb, nq):
    # Mesh2D::ElementMetricCollection::{jacobians, measures, physical_coordinates} (source/Mesh2D.cpp:173-227),
    # LinearFunctional::action (include/LinearFunctional.hpp:145-181), FaceLinearFunctional::action
    # (include/FaceLinearFunctional.hpp:130-164) against the reference's own objects
    r = ref("metrics_lf", spec, nb, nq)
    mesh = product_mesh(spec)
    fem = cb.H1Space(mesh, cb.Basis(nb))
    n, nel = fem.size(), mesh.n_elem()
    assert n == r["ndof"][0] and nel == r["n_elem"][0]
    xq = r["xq"]
    assert np.array_equal(cb.QuadratureRule(nq, cb.GaussLegendre).x(), xq)
    tol = 1e-13
    assert rel(host(fem.element_metrics(xq, "jacobians")).ravel(), r["J"]) < tol
    assert rel(host(fem.element_metrics(xq, "measures")).ravel(), r["detJ"]) < tol
    assert rel(host(fem.element_metrics(xq, "physical_coordinates")).ravel(), r["xphys"]) < tol
    f_mass = lambda x, y: 3.0 * x * x - 2.0 * x * y + y + 1.0
    f_coef = lambda x, y: 1.0 + 0.5 * torch.sin(np.pi * x) * torch.cos(np.pi * y)
    quad = cb.QuadratureRule(nq, cb.GaussLegendre)
    F = torch.full((n,), 3.0, dtype=torch.float64, device="cuda")  # action(f, F) overwrites
    cb.LinearFunctional(fem).action(f_mass, F)
    assert rel(host(F), r["lf_fast"]) < 1e-12
    l2 = cb.LinearFunctional(fem, quad)
    l2.action(f_mass, F)
    assert rel(host(F), r["lf_quad"]) < 1e-12
    l2.action(-0.5, f_coef, F)
    assert rel(host(F), r["lf_quad_acc"]) < 1e-12
    fs = cb.FaceSpace(fem, mesh.boundary_edges())
    assert fs.size() == r["fdof"][0]
    G = torch.full((fs.size(),), -2.0, dtype=torch.float64, device="cuda")
    cb.FaceLinearFunctional(fs).action(f_mass, G)
    assert rel(host(G), r["fl_fast"]) < 1e-12
    fl2 = cb.FaceLinearFunctional(fs, quad)
    fl2.action(f_mass, G)
    assert rel(host(G), r["fl_quad"]) < 1e-12
    fl2.action(1.5, f_coef, G)
    assert rel(host(G), r["fl_quad_acc"]) < 1e-12


@pytest.mark.parametrize("spec,nb,m,maxit,tol", [("file:" + MESH_FILE, 5, 20, 30, 1e-6), ("file:" + MESH_FILE, 4, 200, 60, 1e-4),
                                                 ("rect:16", 4, 30, 30, 1e-6)])
def test_helmholtz_gmres_matches_reference(spec, nb, m, maxit, tol):
    # config 1a: FP64 GMRES(m) on the Helmholtz composite. GMRES(20/30) stagnates on this indefinite problem, so those
    # cases compare the residual history of a fixed number of restart cycles; GMRES(200) (the reference example's m)
    # converges and is compared on iteration count (+-1) and solution.
    omega = 10.0
    r = ref("helm_gmres", spec, nb, omega, m, maxit, tol)
    mesh = product_mesh(spec)
    fem = cb.H1Space(mesh, cb.Basis(nb))
    fs = cb.FaceSpace(fem, mesh.boundary_edges())
    n = fem.size()
    xy = fem.physical_coordinates()
    c = 1.0 + 0.5 * np.sin(np.pi * xy[:, 0]) * np.cos(np.pi * xy[:, 1])
    A = cb.Helmholtz(omega, dev(c * c), dev(c[fs.global_indices()]), fem, fs)
    U = torch.zeros(2 * n, dtype=torch.float64, device="cuda")
    out = cb.gmres(2 * n, U, A, dev(r["b"]), m, maxit, tol)
    assert out.success == bool(r["success"][0])
    ref_it = int(r["num_iter"][0])
    assert abs(out.num_iter - ref_it) <= restart_slack(ref_it), "restarts %d vs reference %d (%s)" % (out.num_iter, ref_it, SPREAD_NOTE)
    k = min(len(out.res_norm), len(r["res_norm"]))
    if out.success:
        assert rel(host(U), r["U"]) < 1e-3
    else:
        assert np.allclose(out.res_norm[:k], r["res_norm"][:k], rtol=1e-6)
        assert rel(host(U), r["U"]) < 1e-6


@pytest.mark.parametrize("nx,nb", [(8, 4), (16, 4), (32, 4), (8, 8), (16, 8)])
def test_ddh_matches_reference(nx, nb):
    # examples/DDH.cpp flow (config 1b and the ladder of SURVEY §8d): index data bit-exact, rhs / one action /
    # postprocess within the FP32 tolerance (bounded by the reference's own run-to-run spread x10, floor 2e-4),
    # GMRES iteration count +-1, solution 1e-3.
    omega = 2 * np.pi * nx / 10
    r = ref("ddh", nx, nb, omega, 20, 100, 1e-4, 2024, timeout=1500)
    mesh = cb.Mesh2D.uniform_rect(nx, -1.0, 1.0, nx, -1.0, 1.0)
    fem = cb.H1Space(mesh, cb.Basis(nb))
    D = cb.DDH(omega, r["a"], fem, nx, nx, 16)
    info = D.info()
    n = D.size()
    assert n == r["n_lambda"][0] and info["n_domains"] == r["n_domains"][0] and info["nt"] == r["nt"][0] and info["dt"] == r["dt"][0]
    # DDH constructor tables, bit for bit (ints) / exactly (floats rounded from the same doubles)
    assert np.array_equal(D.array("B"), r["Bf"])
    assert np.array_equal(D.array("gI"), r["gI"]) and np.array_equal(D.array("sI"), r["sI"])
    assert np.array_equal(D.array("m"), r["m"]) and np.array_equal(D.array("H"), r["H"])
    assert np.array_equal(D.array("a"), r["acoef"]) and np.array_equal(D.array("gmi"), r["gmi"])
    assert np.array_equal(D.array("wh_filter"), r["wh_filter"])
    assert np.allclose(D.array("g"), r["g_tensor"], rtol=2e-7, atol=0)

    spread = rel(r["act_y2"], r["act_y"])  # the reference against itself (shared-memory float atomics)
    tol = max(10 * spread, 2e-4)
    f = dev(r["b"])
    b = torch.empty(n, dtype=torch.float32, device="cuda")
    D.rhs(f, b)
    assert rel(host(b), r["rhs"]) < tol
    y = torch.empty(n, dtype=torch.float32, device="cuda")
    D.action(dev(r["act_x"], torch.float32), y)
    # slots that no subdomain writes hold lambda - (stale memory) in the reference; compare the written ones
    Bout = D.array("B").reshape(info["n_domains"], 2, info["mx_fdof"])[:, 1, :]
    idx = Bout[Bout >= 0]
    mask = np.zeros(n, bool)
    mask[idx] = True
    mask[n // 2 + idx] = True
    assert rel(host(y)[mask], r["act_y"][mask]) < tol, (rel(host(y)[mask], r["act_y"][mask]), spread)

    L = torch.zeros(n, dtype=torch.float32, device="cuda")
    out = cb.gmres(n, L, D, b, 20, 100, 1e-4)
    U = torch.empty(2 * fem.size(), dtype=torch.float64, device="cuda")
    D.postprocess(L, f, U)
    assert out.success == bool(r["success"][0])
    ref_it = int(r["num_iter"][0])
    assert abs(out.num_iter - ref_it) <= restart_slack(ref_it), "restarts %d vs reference %d (%s)" % (out.num_iter, ref_it, SPREAD_NOTE)
    if out.success:
        assert rel(host(U), r["U"]) < 1e-3, rel(host(U), r["U"])
    else:
        # (nx, nb) = (16, 8): the reference itself does not converge (100 restarts, residual stagnating near 0.5 |b|):
        # with omega = 2 pi nx / 10 the 2x2-element subdomains are near a local resonance, the reference's own two
        # consecutive actions differ by 5e-4, and an unconverged, chaotic Krylov history cannot be compared entry by
        # entry. Parity here = same failure, same restart / matvec counts, same first residuals.
        assert out.num_matvec == int(r["num_matvec"][0])
        assert np.allclose(out.res_norm[:2], r["res_norm"][:2], rtol=0.25)
