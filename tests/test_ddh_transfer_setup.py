"""CPU: slot maps of the assembled DDH operator (DDH.transfer_slots, host only) against the reference-layout index map B."""
import numpy as np
import pytest

import cuddhelmholtz_b200 as cb


def _ddh(nx, nb, block):
    mesh = cb.Mesh2D.uniform_rect(nx, -1.0, 1.0, nx, -1.0, 1.0)
    fem = cb.H1Space(mesh, cb.Basis(nb))
    return cb.DDH(10.0, np.ones(fem.size()), fem, nx, nx, block)


@pytest.mark.parametrize("nx,nb,block", [(8, 4, 16), (8, 8, 16), (16, 4, 32), (8, 8, 32), (32, 4, 16)])
def test_transfer_slots_match_B(nx, nb, block):
    d = _ddh(nx, nb, block)
    info = d.info()
    nd, F = info["n_domains"], info["mx_fdof"]
    n = d.size()
    nl = n // 2
    inp, out, orphans = d.transfer_slots()
    assert inp.shape == out.shape == (nd, 2 * F)
    assert (2 * F) % 16 == 0  # 16-byte aligned block columns
    # lambda half and mu half of a face position point at the same pair
    for m in (inp, out):
        assert np.array_equal(m[:, :F] >= 0, m[:, F:] >= 0)
        assert np.array_equal(m[:, F:][m[:, F:] >= 0], nl + m[:, :F][m[:, :F] >= 0])
    B = d.array("B").reshape(nd, 2, F)  # (mx_fdof, 2, dom) column-major
    for m, c in ((inp, 0), (out, 1)):
        s = m[m >= 0]
        assert len(np.unique(s)) == len(s)  # no slot repeats
        b = B[:, c, :]
        b = b[b >= 0]
        assert np.array_equal(np.sort(s), np.sort(np.concatenate([b, nl + b])))
    written = np.zeros(n, bool)
    written[out[out >= 0]] = True
    assert np.array_equal(orphans, np.flatnonzero(~written))
    assert inp.min() >= -1 and out.min() >= -1 and inp.max() < n and out.max() < n


def test_transfer_slots_face_order_is_the_boundary_ring():
    # n_basis 4, block 16 on an 8 x 8 mesh: four subdomains of 13 x 13 DOFs, F = 48 face positions = the boundary ring in ascending
    # grid index Y*13 + X. Subdomain 0 (lower left) has slots on its interface sides X = 12 and Y = 12, end points included, and
    # none on the rest of its physical-boundary sides X = 0, Y = 0.
    d = _ddh(8, 4, 16)
    inp, out, _ = d.transfer_slots()
    n1 = 13
    ring = [at for at in range(n1 * n1) if at % n1 in (0, n1 - 1) or at // n1 in (0, n1 - 1)]
    assert len(ring) == 48
    X = np.array([at % n1 for at in ring])
    Y = np.array([at // n1 for at in ring])
    interface = (X == n1 - 1) | (Y == n1 - 1)
    for m in (inp, out):
        assert np.array_equal(m[0, :48] >= 0, interface)
        assert np.array_equal(m[0, 48:] >= 0, interface)
