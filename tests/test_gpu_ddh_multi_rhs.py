"""GPU: many sources at once on the assembled DDH operator. DDHTransfer.action_batch against row-by-row actions (bitwise, every
transfer-block size, k across the pass boundary), its argument checks, and gmres_batch against sequential MGS gmres solves
(bitwise x, residual history, restart and matvec counts) on a DDHTransfer and on a Python operator."""
import numpy as np
import pytest
import torch

import cuddhelmholtz_b200 as cb
from gpu_util import as_tensor, dev
from test_gpu_ddh_transfer import CASES, SOLVES, _ddh, _recorded_problem

pytestmark = pytest.mark.gpu
KB = 16  # vectors per pass of the batched action kernel
KS = [1, 2, 5, KB, KB + 1, 32]


@pytest.mark.parametrize("nx,nb,block", CASES)
def test_action_batch_rows_are_bitwise_single_actions(nx, nb, block):
    fem, D, f = _ddh(nx, nb, block)
    T = cb.DDHTransfer(D)
    n = T.size()
    orph = torch.as_tensor(D.transfer_slots()[2], dtype=torch.long, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(nx * 100 + nb * 10 + block)
    # rows with a padded stride: only the rows need to be contiguous
    X = (torch.rand((32, n + 5), generator=g, device="cuda") * 2 - 1)[:, :n]
    ref = torch.empty((32, n), device="cuda")
    for j in range(32):
        T.action(X[j], ref[j])
    for k in KS:
        Y = torch.full((k, n), float("nan"), device="cuda")
        c0 = cb.launch_count()
        T.action_batch(X[:k], Y)
        launches = cb.launch_count() - c0
        assert launches <= -(-k // KB) + 1, (k, launches)
        assert torch.equal(Y, ref[:k]), (k, int((Y != ref[:k]).sum()))  # NaN-filled: every slot written, bitwise
        assert torch.equal(Y[:, orph], X[:k, orph])
        Y2 = torch.empty_like(Y)
        T.action_batch(X[:k], Y2)
        assert torch.equal(Y2, Y)


def test_action_batch_rejects_overlap_and_bad_k_and_leaves_y_untouched():
    fem, D, f = _ddh(8, 4, 16)
    T = cb.DDHTransfer(D)
    n = T.size()
    X = torch.rand((33, n), device="cuda")
    Y = torch.full((33, n), 7.0, device="cuda")
    X0, Y0 = X.clone(), Y.clone()
    dup = torch.as_strided(Y, (2, n), (0, 1))           # the same output twice
    half = torch.as_strided(Y, (2, n), (n // 2, 1))     # outputs that overlap by half
    with pytest.raises(cb.CuddhError, match="overlaps output"):
        T.action_batch(X[:2], dup)
    with pytest.raises(cb.CuddhError, match="overlaps output"):
        T.action_batch(X[:2], half)
    with pytest.raises(cb.CuddhError, match="overlaps input"):
        T.action_batch(X[:3], X[1:4])                    # in place / shifted onto the inputs
    with pytest.raises(cb.CuddhError, match="overlaps input"):
        T.action_batch(torch.as_strided(Y, (2, n), (n, 1)), Y[1:3])
    with pytest.raises(cb.CuddhError, match=r"k must be in \[1, 32\]"):
        T.action_batch(X, Y)
    with pytest.raises(cb.CuddhError, match=r"k must be in \[1, 32\]"):
        T.action_batch(X[:0], Y[:0])
    torch.cuda.synchronize()
    assert torch.equal(Y, Y0) and torch.equal(X, X0)


def _sources(fem, omega, centers):
    """(k, 2 ndof) forcings [M g_j; 0] of Gaussian sources g_j at the given centres"""
    xy = fem.physical_coordinates()
    X, Y = xy[:, 0], xy[:, 1]
    n = fem.size()
    s = omega * omega
    F = torch.zeros((len(centers), 2 * n), dtype=torch.float64, device="cuda")
    M = cb.MassMatrix(fem)
    for j, (cx, cy) in enumerate(centers):
        M.action(dev(s / np.pi * np.exp(-s * ((X - cx) ** 2 + (Y - cy) ** 2))), F[j, :n])
    return F


CENTERS = [(-0.5, 0.0), (0.5, -0.5), (0.05, 0.1), (0.8, 0.75), (-0.7, 0.6)]


def _problem(which):
    if which == "recorded128":
        case = next(c for c in SOLVES if c["nx"] == 128)
        fem, D, _ = _recorded_problem(case)
        omega = 2 * np.pi * 128 / 10
    else:  # n_basis 8, smooth slowness (see test_gpu_ddh_transfer.test_transfer_solve_n_basis_8)
        omega = 10.0
        fem, D, _ = _ddh(16, 8, 16, omega, smooth=True)
    return fem, D, _sources(fem, omega, CENTERS)


@pytest.mark.parametrize("which", ["recorded128", "nb8_smooth"])
def test_gmres_batch_is_bitwise_sequential_mgs(which):
    fem, D, F = _problem(which)
    T = cb.DDHTransfer(D)
    n = T.size()
    k0 = len(CENTERS)
    m, maxit, tol = 20, 100, 1e-4
    B = torch.empty((k0, n), device="cuda")
    for j in range(k0):
        T.rhs(F[j], B[j])
    seq = []
    for j in range(k0):
        L = torch.zeros(n, device="cuda")
        o = cb.gmres(n, L, T, B[j], m, maxit, tol, orth=cb.MGS)
        seq.append((o, L))
    # system k0: source 0 again, started from its converged solution (0 iterations while the others run);
    # system k0 + 1: source 1 from the iterate of a 2-restart solve (fewer restarts than from zero)
    Lp = torch.zeros(n, device="cuda")
    cb.gmres(n, Lp, T, B[1], m, 2, tol, orth=cb.MGS)
    X0 = [torch.zeros(n, device="cuda") for _ in range(k0)] + [seq[0][1].clone(), Lp]
    Bs = [B[j] for j in range(k0)] + [B[0], B[1]]
    for j in (k0, k0 + 1):
        L = X0[j].clone()
        seq.append((cb.gmres(n, L, T, Bs[j], m, maxit, tol, orth=cb.MGS), L))
    X = torch.stack(X0)
    outs = cb.gmres_batch(n, X, T, torch.stack(Bs), m, maxit, tol)
    restarts = [o.num_iter for o in outs]
    print("%s: restarts per source %s, matvecs %s" % (which, restarts, [o.num_matvec for o in outs]))
    assert len(set(restarts[:k0])) > 1, restarts  # systems leave the batch at different restarts
    assert outs[k0].success and outs[k0].num_iter == 0 and outs[k0].num_matvec == 1
    for j, (o, L) in enumerate(seq):
        b = outs[j]
        assert (b.success, b.num_iter, b.num_matvec) == (o.success, o.num_iter, o.num_matvec), j
        assert b.res_norm == o.res_norm, j
        assert len(b.time) == len(o.time)
        assert torch.equal(X[j], L), j
    assert all(o.success for o in outs)
    for j in range(k0):
        Ub = torch.empty(F.shape[1], dtype=torch.float64, device="cuda")
        Us = torch.empty_like(Ub)
        T.postprocess(X[j], F[j], Ub)
        T.postprocess(seq[j][1], F[j], Us)
        assert torch.equal(Ub, Us), j


class Stencil:
    """y = -3 x_i + 1.0 x_{i-1} + 1.5 x_{i+1} (FP32), single-vector and column-wise batched forms with the same element arithmetic"""

    def __init__(self, n):
        self.n = n
        self.calls = []  # (input addresses) of every batched call

    @staticmethod
    def _apply(x, y):
        y.copy_(-3.0 * x)
        y[1:] += 1.0 * x[:-1]
        y[:-1] += 1.5 * x[1:]

    def action(self, xp, yp):
        self._apply(as_tensor(xp, self.n, torch.float32), as_tensor(yp, self.n, torch.float32))

    def action_batch(self, xps, yps):
        self.calls.append(list(xps))
        Xc = torch.stack([as_tensor(p, self.n, torch.float32) for p in xps], 1)  # one column per system
        Yc = torch.empty_like(Xc)
        self._apply(Xc, Yc)
        for j, p in enumerate(yps):
            as_tensor(p, self.n, torch.float32).copy_(Yc[:, j])


def test_gmres_batch_python_operator_sees_only_active_systems():
    n, k, m, maxit, tol = 2000, 6, 8, 200, 1e-5
    g = torch.Generator(device="cuda").manual_seed(11)
    B = torch.rand((k, n), generator=g, device="cuda")
    B[2] = 0.0
    B[2, 7] = 1.0  # a point load: converges in fewer restarts than the random ones
    B[4] = torch.linspace(0.0, 1.0, n, device="cuda")
    op = Stencil(n)
    X0 = torch.zeros((k, n), device="cuda")
    cb.gmres(n, X0[1], op, B[1], m, 2, tol, orth=cb.MGS)  # system 1 starts one restart ahead
    cb.gmres(n, X0[3], op, B[3], m, maxit, tol, orth=cb.MGS)  # system 3 starts converged
    seq = []
    for j in range(k):
        L = X0[j].clone()
        seq.append((cb.gmres(n, L, op, B[j], m, maxit, tol, orth=cb.MGS), L))
    X = X0.clone()
    outs = cb.gmres_batch(n, X, op, B, m, maxit, tol)
    for j, (o, L) in enumerate(seq):
        b = outs[j]
        assert (b.success, b.num_iter, b.num_matvec, b.res_norm) == (o.success, o.num_iter, o.num_matvec, o.res_norm), j
        assert torch.equal(X[j], L), j
    restarts = [o.num_iter for o in outs]
    print("stencil: restarts per system %s, batched calls %d, sizes %s" % (restarts, len(op.calls), sorted({len(c) for c in op.calls})))
    assert len(set(restarts)) > 1 and restarts[3] == 0, restarts
    assert all(o.success for o in outs)
    # every system is handed to the operator exactly as often as its own solve applies it, so never after it has left
    assert sum(len(c) for c in op.calls) == sum(o.num_matvec for o in outs)
    assert len(op.calls[0]) == k and min(len(c) for c in op.calls) < k
    xrow = {X[j].data_ptr(): j for j in range(k)}
    for j in range(k):  # x_j is the operator's input once initially and once per restart of its own solve
        assert sum(p == X[j].data_ptr() for c in op.calls for p in c) == 1 + outs[j].num_iter, j
    assert set(p for c in op.calls for p in c if p in xrow) == set(xrow)


def test_gmres_batch_python_operator_exception_aborts_and_is_reraised():
    n = 512

    class Broken(Stencil):
        def action_batch(self, xps, yps):
            if len(self.calls) == 2:
                raise RuntimeError("batched operator exploded")
            super().action_batch(xps, yps)

    B = torch.rand((3, n), device="cuda")
    X = torch.zeros_like(B)
    op = Broken(n)
    with pytest.raises(RuntimeError, match="batched operator exploded"):
        cb.gmres_batch(n, X, op, B, 10, 50, 1e-5)
    assert len(op.calls) == 2
