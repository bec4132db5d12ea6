"""GPU: the assembled DDH interface operator (DDHTransfer) against the WaveHoltz DDH operator it is probed from: bitwise equal
actions on unit vectors, blocks equal to the columns apply_T_range extracts, random inputs, launches per action, and DDH-GMRES
solves with either operator (recorded reference restart counts, the oracle, the n_basis 8 kernels, FGMRES preconditioning)."""
import json
import os

import numpy as np
import pytest
import torch

import cuddhelmholtz_b200 as cb
from conftest import GOLD
from gpu_util import dev, host, rel
from oracle import ops as O
from test_gpu_parity import _ddh_pair

pytestmark = pytest.mark.gpu
SOLVES = json.load(open(os.path.join(GOLD, "reference_ddh_solves.json")))["solves"]


def _ddh(nx, nb, block, omega=10.0, smooth=False):
    """library DDH with the variable coefficient of test_gpu_parity._ddh_pair (smooth=True: the smooth slowness of
    test_gpu_parity.test_ddh_preconditioned_fgmres), and its Gaussian-source forcing"""
    mesh = cb.Mesh2D.uniform_rect(nx, -1.0, 1.0, nx, -1.0, 1.0)
    fem = cb.H1Space(mesh, cb.Basis(nb))
    xy = fem.physical_coordinates()
    X, Y = xy[:, 0], xy[:, 1]
    if smooth:
        ha = 1.0 + 0.25 * np.exp(-8.0 * (X * X + Y * Y))
    else:
        ha = np.where(X * X + Y * Y < 0.0625, 0.2, 1.0) + 0.05 * np.sin(3 * X)
    D = cb.DDH(omega, ha, fem, nx, nx, block)
    s = omega * omega
    src = s / np.pi * np.exp(-s * ((X + 0.5) ** 2 + Y ** 2)) + s / np.pi * np.exp(-s * ((X - 0.5) ** 2 + (Y + 0.5) ** 2))
    f = torch.zeros(2 * fem.size(), dtype=torch.float64, device="cuda")
    cb.MassMatrix(fem).action(dev(src), f[:fem.size()])
    return fem, D, f


CASES = [(8, 4, 16), (8, 8, 16), (16, 4, 32), (8, 8, 32), (16, 4, 16)]


@pytest.mark.parametrize("nx,nb,block", CASES)
def test_transfer_is_bitwise_the_ddh_action_on_unit_vectors(nx, nb, block):
    fem, D, f = _ddh(nx, nb, block)
    T = cb.DDHTransfer(D)
    n = D.size()
    info = T.info()
    nd, tf = info["n_domains"], info["two_f"]
    assert info["block_bytes"] == nd * tf * tf * 4
    assert info["probe_launches"] >= 2 * tf
    slots = np.arange(n) if n <= 600 else np.sort(np.random.default_rng(7).choice(n, 200, replace=False))
    e = torch.zeros(n, dtype=torch.float32, device="cuda")
    y0 = torch.empty_like(e)
    y1 = torch.empty_like(e)
    bad = []
    for s in slots:
        e[s] = 1.0
        D.action(e, y0)
        T.action(e, y1)
        e[s] = 0.0
        if not torch.equal(y0, y1):
            bad.append(int(s))
    assert not bad, bad[:10]
    # blocks: column k of M_p = the WaveHoltz kernel's response of subdomain p alone to a 1 at its input k
    inp, out, _ = D.transfer_slots()
    t = torch.empty_like(e)
    for p in (0, nd - 1):
        M = T.block(p)
        ref = np.zeros((tf, tf), np.float32)
        for k in range(tf):
            if inp[p, k] < 0:
                continue
            e[inp[p, k]] = 1.0
            D.apply_T_range(e, t, p, p + 1)
            e[inp[p, k]] = 0.0
            th = host(t)
            w = out[p] >= 0
            ref[w, k] = th[out[p][w]]
        assert np.array_equal(M, ref), (p, np.abs(M - ref).max())


@pytest.mark.parametrize("nx,nb,block", CASES)
def test_transfer_random_input(nx, nb, block):
    fem, D, f = _ddh(nx, nb, block)
    T = cb.DDHTransfer(D)
    n = D.size()
    _, _, orphans = D.transfer_slots()
    lam = np.random.default_rng(2024).uniform(-1, 1, n).astype(np.float32)
    lam[orphans] = 0.0
    x = dev(lam, torch.float32)
    y0 = torch.empty_like(x)
    D.action(x, y0)
    y1 = torch.empty_like(x)
    c0 = cb.launch_count()
    T.action(x, y1)
    launches = cb.launch_count() - c0
    assert launches <= 2, launches
    y2 = torch.empty_like(x)
    T.action(x, y2)
    assert torch.equal(y1, y2)  # deterministic
    e = rel(host(y1), host(y0))
    print("nx %d n_basis %d block %d: rel(transfer, WaveHoltz) = %.3e, %d launch(es) per action, nt = %d"
          % (nx, nb, block, e, launches, D.info()["nt"]))
    assert e < 2e-4, e


def test_transfer_launches_do_not_depend_on_nt():
    counts = []
    for omega in (5.0, 40.0):
        fem, D, f = _ddh(8, 4, 16, omega)
        T = cb.DDHTransfer(D)
        x = torch.ones(D.size(), dtype=torch.float32, device="cuda")
        y = torch.empty_like(x)
        c0 = cb.launch_count()
        T.action(x, y)
        counts.append((D.info()["nt"], cb.launch_count() - c0))
    assert counts[0][0] != counts[1][0] and counts[0][1] == counts[1][1] <= 2, counts


def _recorded_problem(case):
    """the discrete problem of tests/test_gpu_reference_recorded.py (examples/DDH.cpp flow)"""
    nx, nb = case["nx"], case["n_basis"]
    omega = 2 * np.pi * nx / 10
    mesh = cb.Mesh2D.uniform_rect(nx, -1.0, 1.0, nx, -1.0, 1.0)
    fem = cb.H1Space(mesh, cb.Basis(nb))
    n = fem.size()
    s = omega * omega
    f_src = lambda X, Y: s / np.pi * torch.exp(-s * ((X + 0.5) ** 2 + Y ** 2)) + s / np.pi * torch.exp(-s * ((X - 0.5) ** 2 + (Y + 0.5) ** 2))
    f_alpha = lambda X, Y: torch.where(X * X + Y * Y < 0.0625, torch.full_like(X, 0.2), torch.full_like(X, 1.0))
    f = torch.zeros(2 * n, dtype=torch.float64, device="cuda")
    lf = cb.LinearFunctional(fem)
    lf.action(f_src, f[:n])
    la = torch.empty(n, dtype=torch.float64, device="cuda")
    lf.action(f_alpha, la)
    a = torch.empty_like(la)
    cb.DiagInvMassMatrix(fem).action(la, a)
    return fem, cb.DDH(omega, a.cpu().numpy(), fem, nx, nx, 16), f


@pytest.mark.parametrize("case", SOLVES, ids=lambda c: "nx%d" % c["nx"])
def test_transfer_solve_matches_recorded_reference(case):
    fem, D, f = _recorded_problem(case)
    T = cb.DDHTransfer(D)
    m = T.size()
    b = torch.empty(m, dtype=torch.float32, device="cuda")
    T.rhs(f, b)
    L = torch.zeros(m, dtype=torch.float32, device="cuda")
    out = cb.gmres(m, L, T, b, case["m"], case["maxit"], case["tol"], orth=cb.MGS)
    print("nx %d: transfer operator %d restarts, reference %d" % (case["nx"], out.num_iter, case["restarts"]))
    assert out.success == case["success"]
    assert abs(out.num_iter - case["restarts"]) <= 1, (out.num_iter, case["restarts"])
    U = torch.empty(f.numel(), dtype=torch.float64, device="cuda")
    T.postprocess(L, f, U)
    assert bool(torch.isfinite(U).all()) and float(U.norm()) > 0


def test_transfer_solve_matches_oracle_config_1b():
    omega = 10.0
    ofem, pfem, oD, pD, f = _ddh_pair(8, 4, omega)
    T = cb.DDHTransfer(pD)
    n = T.size()
    df = dev(f)
    b = torch.empty(n, dtype=torch.float32, device="cuda")
    T.rhs(df, b)
    L = torch.zeros(n, dtype=torch.float32, device="cuda")
    out = cb.gmres(n, L, T, b, 20, 100, 1e-4)
    U = torch.empty(2 * ofem.ndof, dtype=torch.float64, device="cuda")
    T.postprocess(L, df, U)
    Lo = np.zeros(n, np.float32)
    oo = O.gmres(n, Lo, oD.action, oD.rhs(f), 20, 100, 1e-4, dtype=np.float32)
    assert out.success and oo["success"]
    assert abs(out.num_iter - oo["num_iter"]) <= 1, (out.num_iter, oo["num_iter"])
    assert rel(host(U), oD.postprocess(Lo, f)) < 1e-3


@pytest.mark.parametrize("nx,block", [(8, 16), (16, 16), (8, 32), (16, 32)])
def test_transfer_solve_n_basis_8(nx, block):
    # smooth coefficient: with the 0.2 / 1.0 jump of _ddh_pair, n_basis 8 at nx 16 puts the subdomain time stepping into its
    # unstable range (|T x| ~ 1e10 |x|, the FP32 WaveHoltz action linear to only ~1e-3; the oracle shows the same), where GMRES on
    # the WaveHoltz operator stagnates and there is no restart count to compare with
    fem, D, f = _ddh(nx, 8, block, smooth=True)
    T = cb.DDHTransfer(D)
    n = D.size()
    b = torch.empty(n, dtype=torch.float32, device="cuda")
    D.rhs(f, b)
    res = []
    for op in (D, T):
        L = torch.zeros(n, dtype=torch.float32, device="cuda")
        out = cb.gmres(n, L, op, b, 20, 100, 1e-4)
        U = torch.empty(f.numel(), dtype=torch.float64, device="cuda")
        op.postprocess(L, f, U)
        res.append((out, U))
    (o0, U0), (o1, U1) = res
    print("nx %d block %d: WaveHoltz %d restarts, transfer %d" % (nx, block, o0.num_iter, o1.num_iter))
    assert o0.success == o1.success
    assert abs(o0.num_iter - o1.num_iter) <= 1, (o0.num_iter, o1.num_iter)
    assert rel(host(U1), host(U0)) < 1e-3, rel(host(U1), host(U0))


def test_transfer_as_fgmres_preconditioner():
    # the set-up of test_gpu_parity.test_ddh_preconditioned_fgmres, with the DDH inside the preconditioner swapped for its
    # assembled form: same outer iteration count (+-1)
    nx, nb = 16, 4
    omega = 2 * np.pi * nx / 10
    mesh = cb.Mesh2D.uniform_rect(nx, -1.0, 1.0, nx, -1.0, 1.0)
    fem = cb.H1Space(mesh, cb.Basis(nb))
    fs = cb.FaceSpace(fem, mesh.boundary_edges())
    n = fem.size()
    xy = fem.physical_coordinates()
    X, Y = xy[:, 0], xy[:, 1]
    ha = 1.0 + 0.25 * np.exp(-8.0 * (X * X + Y * Y))
    A = cb.Helmholtz(omega, dev(ha * ha), dev(ha[fs.global_indices()]), fem, fs)
    s = omega * omega
    src = s / np.pi * np.exp(-s * ((X + 0.5) ** 2 + Y ** 2))
    b = torch.zeros(2 * n, dtype=torch.float64, device="cuda")
    cb.MassMatrix(fem).action(dev(src), b[:n])
    D = cb.DDH(omega, ha, fem, nx, nx, 16)
    outs = []
    for op in (D, cb.DDHTransfer(D)):
        P = cb.DDHPreconditioner(op, m=20, maxit=100, tol=1e-5)
        U = torch.zeros(2 * n, dtype=torch.float64, device="cuda")
        o = cb.gmres(2 * n, U, A, b, 30, 3, 1e-8, P=P, flexible=True)
        Ax = torch.empty_like(b)
        A.action(U, Ax)
        assert o.success and float((Ax - b).norm() / b.norm()) < 1.01e-8
        outs.append(o)
    print("FGMRES outer matvecs: WaveHoltz preconditioner %d, transfer preconditioner %d" % (outs[0].num_matvec, outs[1].num_matvec))
    assert abs(outs[0].num_iter - outs[1].num_iter) <= 1
    assert abs(outs[0].num_matvec - outs[1].num_matvec) <= 1, (outs[0].num_matvec, outs[1].num_matvec)


def test_transfer_out_of_memory_names_the_bytes_and_leaves_the_ddh_usable():
    fem, D, f = _ddh(8, 4, 16)
    with pytest.raises(cb.CuddhError, match=r"needs \d+ bytes"):
        cb.DDHTransfer(D, max_bytes=1)
    n = D.size()
    b = torch.empty(n, dtype=torch.float32, device="cuda")
    D.rhs(f, b)
    L = torch.zeros(n, dtype=torch.float32, device="cuda")
    out = cb.gmres(n, L, D, b, 20, 100, 1e-4)
    assert out.success
