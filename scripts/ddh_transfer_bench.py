"""Assembled DDH operator (DDHTransfer) against the WaveHoltz DDH operator on one GPU, examples/DDH.cpp flow (uniform_rect(nx),
omega = 2 pi nx / 10, FP32 GMRES(20), maxit 100, tol 1e-4, x0 = 0, subdomain block 16). Per case one JSON line:
  probe_ms                  creation of the transfer handle (2F WaveHoltz actions + scatter / gather), CUDA events
  transfer_action_ms        median CUDA-event time of single actions after warm-up; GB/s from the modelled bytes per action (blocks,
                            slot maps, gathered / written vector entries) and its share of the 6459 GB/s measured copy peak
  wh_action_ms              median CUDA-event time of the WaveHoltz action
  *_solve_s, *_restarts     end-to-end DDH-GMRES wall time (rhs + solve, and for the transfer operator its probing), restart counts
  solution_rel              ||u_transfer - u_wh|| / ||u_wh|| of the postprocessed solutions
  action_rel_diff, wh_gain  the two actions on one random input, and |T x| / |x| of the WaveHoltz map for it
The first line records the GPU name and power limit read in the same run.
usage: python scripts/ddh_transfer_bench.py [--cases 128:4,512:4,256:8] [--reps 30] [--max-seconds 600] [--out file.jsonl]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

COPY_PEAK_GBS = 6459.0
L2_BYTES = 126 * 1024 * 1024


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clk = [s.strip() for s in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def median_ms(torch, fn, reps, warmup):
    for _ in range(warmup):
        fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    t = sorted(a.elapsed_time(b) for a, b in ev)
    return t[len(t) // 2]


def problem(cb, torch, np, nx, nb):
    """the discrete problem of examples/DDH.cpp (load on the first block, coefficient projected with diag(M)^-1)"""
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
    torch.cuda.synchronize()
    return fem, cb.DDH(omega, a.cpu().numpy(), fem, nx, nx, 16), f


def solve(cb, torch, op, f, n_u, max_seconds, make=None):
    """rhs + GMRES (+ creating the operator with `make`), synchronised wall time"""
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if make is not None:
        op = make()
    m = op.size()
    b = torch.empty(m, dtype=torch.float32, device="cuda")
    op.rhs(f, b)
    L = torch.zeros(m, dtype=torch.float32, device="cuda")
    out = cb.gmres(m, L, op, b, 20, 100, 1e-4, orth=cb.MGS, max_seconds=max_seconds)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    U = torch.empty(n_u, dtype=torch.float64, device="cuda")
    op.postprocess(L, f, U)
    return op, out, dt, U


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="128:4,512:4,256:8", help="nx:n_basis,...")
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--max-seconds", type=float, default=600.0, help="time box of each GMRES solve")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()

    import numpy as np
    import torch
    import cuddhelmholtz_b200 as cb

    if not torch.cuda.is_available():
        raise SystemExit("ddh_transfer_bench.py measures on a GPU; none is visible")
    lines = [dict(gpu_identity(), torch_device=torch.cuda.get_device_name(0))]
    print(json.dumps(lines[0]), flush=True)
    for case in args.cases.split(","):
        nx, nb = (int(v) for v in case.split(":"))
        fem, D, f = problem(cb, torch, np, nx, nb)
        n_u = 2 * fem.size()
        # WaveHoltz operator: action and end-to-end solve
        n = D.size()
        x = torch.randn(n, dtype=torch.float32, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
        y = torch.empty_like(x)
        wh_ms = median_ms(torch, lambda: D.action(x, y), max(5, args.reps // 3), 2)
        _, o_wh, t_wh, U_wh = solve(cb, torch, D, f, n_u, args.max_seconds)
        # assembled operator: end-to-end solve with its probing, then the action on its own
        T, o_tr, t_tr, U_tr = solve(cb, torch, None, f, n_u, args.max_seconds, make=lambda: cb.DDHTransfer(D))
        info = T.info()
        tr_ms = median_ms(torch, lambda: T.action(x, y), args.reps, 5)
        y_wh = torch.empty_like(x)
        D.action(x, y_wh)
        T.action(x, y)
        gbs = info["bytes_per_action"] / (tr_ms * 1e-3) / 1e9
        line = {
            "nx": nx, "n_basis": nb, "block": 16, "n_domains": info["n_domains"], "two_f": info["two_f"], "nt": D.info()["nt"],
            "kernel_kind": D.kernel_kind(),
            "block_bytes": info["block_bytes"], "bytes_per_action": info["bytes_per_action"],
            "blocks_fit_l2": info["block_bytes"] < L2_BYTES,
            "probe_ms": info["probe_ms"], "probe_launches": info["probe_launches"],
            "transfer_action_ms": tr_ms, "transfer_action_GBs": gbs, "transfer_action_copy_peak_frac": gbs / COPY_PEAK_GBS,
            "wh_action_ms": wh_ms, "action_speedup": wh_ms / tr_ms,
            "action_rel_diff": float((y - y_wh).norm() / y_wh.norm()),
            "wh_gain": float((x - y_wh).norm() / x.norm()),  # |T x| / |x| of the random input: >> 1 = unstable local time stepping
            "wh_solve_s": t_wh, "wh_restarts": o_wh.num_iter, "wh_matvecs": o_wh.num_matvec, "wh_success": o_wh.success,
            "transfer_solve_s": t_tr, "transfer_restarts": o_tr.num_iter, "transfer_matvecs": o_tr.num_matvec,
            "transfer_success": o_tr.success, "solve_speedup": t_wh / t_tr,
            "solution_rel": float((U_tr - U_wh).norm() / U_wh.norm()),
            "action_reps": args.reps, "solve_max_seconds": args.max_seconds,
        }
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
