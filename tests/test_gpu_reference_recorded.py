"""GPU: DDH-GMRES solves of the examples/DDH.cpp flow (oracle/ref_driver.cu cmd_ddh) against the outcome the UNMODIFIED reference
library recorded for the same problems (tests/golden/reference_ddh_solves.json: success and restart count). Unlike
tests/test_gpu_reference.py this needs no build of the reference, so it runs wherever the library does."""
import json
import os

import numpy as np
import pytest
import torch

import cuddhelmholtz_b200 as cb
from conftest import GOLD

pytestmark = pytest.mark.gpu
SOLVES = json.load(open(os.path.join(GOLD, "reference_ddh_solves.json")))["solves"]


@pytest.mark.parametrize("case", SOLVES, ids=lambda c: "nx%d" % c["nx"])
def test_ddh_example_solve_matches_recorded_reference(case):
    nx, nb = case["nx"], case["n_basis"]
    omega = 2 * np.pi * nx / 10
    mesh = cb.Mesh2D.uniform_rect(nx, -1.0, 1.0, nx, -1.0, 1.0)
    fem = cb.H1Space(mesh, cb.Basis(nb))
    n = fem.size()
    # the discrete problem of the recorded runs (oracle/ref_driver.cu cmd_ddh): load (f_src, phi_i) on the first block, coefficient
    # alpha projected as diag(M)^-1 (alpha, phi_i), both with the collocated Gauss-Lobatto rule of LinearFunctional(fem)
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
    ha = a.cpu().numpy()
    D = cb.DDH(omega, ha, fem, nx, nx, 16)
    m = D.size()
    b = torch.empty(m, dtype=torch.float32, device="cuda")
    D.rhs(f, b)
    L = torch.zeros(m, dtype=torch.float32, device="cuda")
    out = cb.gmres(m, L, D, b, case["m"], case["maxit"], case["tol"], orth=cb.MGS)
    assert out.success == case["success"]
    # +-1 restart: the reference's own count varies by one from run to run (FP32 shared-memory atomics in its DDH kernel)
    assert abs(out.num_iter - case["restarts"]) <= 1, (out.num_iter, case["restarts"])
    U = torch.empty(2 * n, dtype=torch.float64, device="cuda")
    D.postprocess(L, f, U)
    assert bool(torch.isfinite(U).all()) and float(U.norm()) > 0
