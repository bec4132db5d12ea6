"""Many sources on one assembled DDH operator (DDHTransfer), examples/DDH.cpp flow (uniform_rect(nx), omega = 2 pi nx / 10, FP32
GMRES(20), maxit 100, tol 1e-4, x0 = 0, subdomain block 16). For every case and k in --ks, one JSON line each for:
  kind "action"   the batched action on k random vectors against k single actions: median CUDA-event time after warm-up, GB/s from
                  the block bytes streamed (once per pass of 16 vectors) and FP32 FLOP/s from 2 (2F)^2 n_domains k
  kind "solve"    k Gaussian sources at k distinct seeded positions (--solve-cases only): one probe, k rhs, one gmres_batch and k
                  postprocess, against the same DDHTransfer with k sequential gmres calls (orth MGS); synchronised wall times
                  split into rhs + postprocess (2 WaveHoltz runs per source) and solve; restart counts per source, and whether the
                  batched solutions, residual histories and counts are bitwise those of the sequential solves
The first line records the GPU name and power limit read in the same run.
usage: python scripts/ddh_multi_rhs_bench.py [--cases 128:4,512:4,256:8] [--solve-cases 128:4,512:4] [--ks 1,4,8,16,32]
                                              [--reps 30] [--out file.jsonl]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from ddh_transfer_bench import gpu_identity, median_ms  # noqa: E402

KB = 16  # vectors per pass of the batched action kernel


def problem(cb, torch, np, nx, nb):
    """operator of examples/DDH.cpp (coefficient projected with diag(M)^-1) and a source builder for it"""
    omega = 2 * np.pi * nx / 10
    mesh = cb.Mesh2D.uniform_rect(nx, -1.0, 1.0, nx, -1.0, 1.0)
    fem = cb.H1Space(mesh, cb.Basis(nb))
    n = fem.size()
    s = omega * omega
    lf = cb.LinearFunctional(fem)
    f_alpha = lambda X, Y: torch.where(X * X + Y * Y < 0.0625, torch.full_like(X, 0.2), torch.full_like(X, 1.0))
    la = torch.empty(n, dtype=torch.float64, device="cuda")
    lf.action(f_alpha, la)
    a = torch.empty_like(la)
    cb.DiagInvMassMatrix(fem).action(la, a)
    torch.cuda.synchronize()
    D = cb.DDH(omega, a.cpu().numpy(), fem, nx, nx, 16)

    def sources(centers):
        F = torch.zeros((len(centers), 2 * n), dtype=torch.float64, device="cuda")
        for j, (cx, cy) in enumerate(centers):
            lf.action(lambda X, Y: s / np.pi * torch.exp(-s * ((X - cx) ** 2 + (Y - cy) ** 2)), F[j, :n])
        return F

    return fem, D, sources


def action_line(cb, torch, T, k, reps):
    info = T.info()
    n = T.size()
    g = torch.Generator(device="cuda").manual_seed(k)
    X = torch.rand((k, n), generator=g, device="cuda") * 2 - 1
    Y = torch.empty_like(X)
    Ys = torch.empty_like(X)

    def singles():
        for j in range(k):
            T.action(X[j], Ys[j])

    c0 = cb.launch_count()
    T.action_batch(X, Y)
    launches = cb.launch_count() - c0
    t_batch = median_ms(torch, lambda: T.action_batch(X, Y), reps, 5)
    t_single = median_ms(torch, singles, max(5, reps // 2), 2)
    singles()
    T.action_batch(X, Y)
    torch.cuda.synchronize()
    passes = -(-k // KB)
    flops = 2.0 * info["two_f"] ** 2 * info["n_domains"] * k
    return {
        "kind": "action", "k": k, "launches": launches, "passes": passes,
        "batch_ms": t_batch, "singles_ms": t_single, "speedup": t_single / t_batch,
        "batch_ms_per_vector": t_batch / k, "single_ms": t_single / k,
        "batch_block_GBs": info["block_bytes"] * passes / (t_batch * 1e-3) / 1e9,
        "batch_TFLOPs": flops / (t_batch * 1e-3) / 1e12,
        "single_block_GBs": info["block_bytes"] * k / (t_single * 1e-3) / 1e9,
        "bitwise_rows": bool(torch.equal(Y, Ys)), "reps": reps,
    }


def solve_line(cb, torch, np, T, fem, sources, k, probe_ms):
    n = T.size()
    rng = np.random.default_rng(1000 + k)
    centers = [tuple(c) for c in rng.uniform(-0.8, 0.8, (k, 2))]
    F = sources(centers)
    n_u = F.shape[1]
    m, maxit, tol = 20, 100, 1e-4

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        return r, time.perf_counter() - t0

    def rhs_all(B):
        for j in range(k):
            T.rhs(F[j], B[j])

    def post_all(L, U):
        for j in range(k):
            T.postprocess(L[j], F[j], U[j])

    # batched
    Bb = torch.empty((k, n), device="cuda")
    Lb = torch.zeros((k, n), device="cuda")
    Ub = torch.empty((k, n_u), dtype=torch.float64, device="cuda")
    _, tb_rhs = timed(lambda: rhs_all(Bb))
    outs, tb_solve = timed(lambda: cb.gmres_batch(n, Lb, T, Bb, m, maxit, tol))
    _, tb_post = timed(lambda: post_all(Lb, Ub))
    # sequential
    Bs = torch.empty((k, n), device="cuda")
    Ls = torch.zeros((k, n), device="cuda")
    Us = torch.empty((k, n_u), dtype=torch.float64, device="cuda")
    _, ts_rhs = timed(lambda: rhs_all(Bs))
    seq, ts_solve = timed(lambda: [cb.gmres(n, Ls[j], T, Bs[j], m, maxit, tol, orth=cb.MGS) for j in range(k)])
    _, ts_post = timed(lambda: post_all(Ls, Us))
    bitwise = bool(torch.equal(Lb, Ls)) and all(
        (a.num_iter, a.num_matvec, a.res_norm, a.success) == (b.num_iter, b.num_matvec, b.res_norm, b.success) for a, b in zip(outs, seq))
    tb = probe_ms * 1e-3 + tb_rhs + tb_solve + tb_post
    ts = probe_ms * 1e-3 + ts_rhs + ts_solve + ts_post
    return {
        "kind": "solve", "k": k, "probe_s": probe_ms * 1e-3,
        "batch_rhs_post_s": tb_rhs + tb_post, "batch_solve_s": tb_solve, "batch_total_s": tb,
        "seq_rhs_post_s": ts_rhs + ts_post, "seq_solve_s": ts_solve, "seq_total_s": ts,
        "solve_speedup": ts_solve / tb_solve, "total_speedup": ts / tb,
        "batch_solve_s_per_source": tb_solve / k, "seq_solve_s_per_source": ts_solve / k,
        "restarts": [o.num_iter for o in outs], "matvecs": [o.num_matvec for o in outs], "success": [o.success for o in outs],
        "bitwise_equal_to_sequential": bitwise,
        "solution_max_abs_diff": float((Ub - Us).abs().max()),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="128:4,512:4,256:8", help="nx:n_basis,... (batched action)")
    ap.add_argument("--solve-cases", default="128:4,512:4", help="nx:n_basis,... also solved end to end")
    ap.add_argument("--ks", default="1,4,8,16,32")
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()

    import numpy as np
    import torch
    import cuddhelmholtz_b200 as cb

    if not torch.cuda.is_available():
        raise SystemExit("ddh_multi_rhs_bench.py measures on a GPU; none is visible")
    ks = [int(v) for v in args.ks.split(",")]
    solve_cases = set(args.solve_cases.split(",")) if args.solve_cases else set()
    lines = [dict(gpu_identity(), torch_device=torch.cuda.get_device_name(0))]
    print(json.dumps(lines[0]), flush=True)
    for case in args.cases.split(","):
        nx, nb = (int(v) for v in case.split(":"))
        fem, D, sources = problem(cb, torch, np, nx, nb)
        T = cb.DDHTransfer(D)
        info = T.info()
        head = {"nx": nx, "n_basis": nb, "block": 16, "n_domains": info["n_domains"], "two_f": info["two_f"], "n": T.size(),
                "block_bytes": info["block_bytes"], "probe_ms": info["probe_ms"]}
        for k in ks:
            line = dict(head, **action_line(cb, torch, T, k, args.reps))
            lines.append(line)
            print(json.dumps(line), flush=True)
        if case in solve_cases:
            for k in ks:
                line = dict(head, **solve_line(cb, torch, np, T, fem, sources, k, info["probe_ms"]))
                lines.append(line)
                print(json.dumps(line), flush=True)
        del T, D
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as fh:
            fh.write("".join(json.dumps(l) + "\n" for l in lines))


if __name__ == "__main__":
    main()
