"""GPU: the DDH kernels that the default configuration does not reach - ddh_kernel<NB, NEL> under CUDDH_B200_DDH_V1 (instead of
the register-tiled kernels), and the per-element metric branch (g_uniform = 0) that a structured but warped mesh takes -
against the oracle (oracle/ops.py DDH) at the tolerance of test_gpu_parity.test_ddh_rhs_action_postprocess, and the
assembled operator DDHTransfer over such a handle."""
import numpy as np
import pytest
import torch

import cuddhelmholtz_b200 as cb
from gpu_util import dev, host, rel, warped_mesh
from oracle import ops as O
from oracle import setup_np as S
from test_gpu_parity import _ddh_pair

pytestmark = pytest.mark.gpu
TOL = 2e-4


def _written(oD):
    """slots some subdomain writes (the others, orphans, are zero in rhs and must be zero in lambda)"""
    w = np.zeros(oD.size, bool)
    Bo = oD.d.B[:, 1, :]
    w[Bo[Bo >= 0]] = True
    w[oD.n_lambda + Bo[Bo >= 0]] = True
    return w


def _check_against_oracle(ofem, oD, pD, f):
    """rhs, action (bitwise repeatable) and postprocess of the library handle against the oracle; returns lambda"""
    n = pD.size()
    assert n == oD.size
    df = dev(f)
    b = torch.full((n,), 3.0, dtype=torch.float32, device="cuda")
    pD.rhs(df, b)
    assert rel(host(b), oD.rhs(f)) < TOL, rel(host(b), oD.rhs(f))
    w = _written(oD)
    assert np.all(host(b)[~w] == 0.0)
    lam = np.random.default_rng(2024).uniform(-1, 1, n).astype(np.float32)
    lam[~w] = 0.0
    y = torch.empty(n, dtype=torch.float32, device="cuda")
    pD.action(dev(lam, torch.float32), y)
    yo = oD.action(lam)
    assert rel(host(y), yo) < TOL, rel(host(y), yo)
    y2 = torch.full((n,), 9.0, dtype=torch.float32, device="cuda")
    pD.action(dev(lam, torch.float32), y2)
    assert torch.equal(y, y2)
    u = torch.empty(2 * ofem.ndof, dtype=torch.float64, device="cuda")
    pD.postprocess(dev(lam, torch.float32), df, u)
    uo = oD.postprocess(lam, f)
    assert rel(host(u), uo) < TOL, rel(host(u), uo)
    return lam, host(y)


@pytest.mark.parametrize("nx,nb,block", [(8, 4, 16), (4, 8, 16), (16, 4, 32), (8, 8, 32)])
def test_ddh_v1_kernels_match_oracle_and_register_tiled(nx, nb, block, monkeypatch):
    monkeypatch.delenv("CUDDH_B200_DDH_V1", raising=False)
    ofem, pfem, oD, pD_tiled, f = _ddh_pair(nx, nb, 10.0, block)
    monkeypatch.setenv("CUDDH_B200_DDH_V1", "1")
    ha = np.where((ofem.xy ** 2).sum(1) < 0.0625, 0.2, 1.0) + 0.05 * np.sin(3 * ofem.xy[:, 0])
    pD = cb.DDH(10.0, ha, pfem, nx, nx, block)
    monkeypatch.delenv("CUDDH_B200_DDH_V1")
    assert pD.kernel_kind() == 0
    lam, y = _check_against_oracle(ofem, oD, pD, f)
    # the same problem on the default handle (register-tiled where it applies)
    yt = torch.empty(pD.size(), dtype=torch.float32, device="cuda")
    pD_tiled.action(dev(lam, torch.float32), yt)
    assert rel(y, host(yt)) < TOL, rel(y, host(yt))


@pytest.mark.parametrize("nx,nb,block", [(16, 4, 16), (16, 8, 32)])
def test_ddh_per_element_metric_on_a_warped_mesh(nx, nb, block, monkeypatch):
    monkeypatch.delenv("CUDDH_B200_DDH_V1", raising=False)
    xy, el = warped_mesh(nx)
    om = S.mesh_from_vertices(xy, el)
    ofem = O.H1(om, nb)
    pfem = cb.H1Space(cb.Mesh2D.from_vertices(xy, el), cb.Basis(nb))
    assert np.array_equal(pfem.global_indices().ravel(), ofem.I)
    X, Y = ofem.xy[:, 0], ofem.xy[:, 1]
    # smooth slowness: with the 0.2 / 1.0 jump of _ddh_pair, n_basis 8 at nx 16 is the regime where the FP32 subdomain time
    # stepping amplifies by about 1e10 (DESIGN §5.1) and no FP32 operator can match the oracle
    ha = 1.0 + 0.25 * np.exp(-8.0 * (X * X + Y * Y))
    omega = 10.0
    oD = O.DDH(omega, ha, ofem, nx, nx, block)
    pD = cb.DDH(omega, ha, pfem, nx, nx, block)
    info = pD.info()
    assert info["nt"] == oD.d.nt and info["dt"] == oD.d.dt
    assert pD.kernel_kind() == 0
    # the per-element metric really differs between elements (otherwise the uniform branch would serve this mesh)
    g = pD.array("g").reshape(-1, 3 * nb * nb)
    assert np.abs(g - g[0]).max() > 1e-3 * np.abs(g).max()
    s = omega * omega
    src = s / np.pi * np.exp(-s * ((X + 0.5) ** 2 + Y ** 2)) + s / np.pi * np.exp(-s * ((X - 0.5) ** 2 + (Y + 0.5) ** 2))
    f = np.concatenate([O.MassMatrix(ofem).action(src), np.zeros(ofem.ndof)])
    _check_against_oracle(ofem, oD, pD, f)


def test_transfer_over_a_v1_handle_is_bitwise_its_action(monkeypatch):
    monkeypatch.setenv("CUDDH_B200_DDH_V1", "1")
    ofem, pfem, oD, pD, f = _ddh_pair(8, 4, 10.0, 16)
    monkeypatch.delenv("CUDDH_B200_DDH_V1")
    assert pD.kernel_kind() == 0
    T = cb.DDHTransfer(pD)
    n = pD.size()
    e = torch.zeros(n, dtype=torch.float32, device="cuda")
    y0, y1 = torch.empty_like(e), torch.empty_like(e)
    for s in np.random.default_rng(5).choice(n, 24, replace=False):
        e[s] = 1.0
        pD.action(e, y0)
        T.action(e, y1)
        e[s] = 0.0
        assert torch.equal(y0, y1), int(s)
