#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (BASELINE.json: "DDH-GMRES solve time & GDOF/s operator apply at 1/2/4/8
B200 vs %HBM roofline").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

value / e2e / roofline  (BASELINE configs[1]): operator apply on a synthetic structured 1024x1024 quad mesh, n_basis 5
    (degree 4): one "step" is one Helmholtz composite action (stiffness + weighted mass on u and v, boundary face mass) on
    [u; v], GDOF/s = 2*ndof / time, next to the fraction of the measured HBM roofline of the dominant kernel.
    N > 1 (launched by torch.distributed.run): weak scaling, one 1024x1024 slab per rank, interface rows exchanged between
    neighbouring ranks (cuddhelmholtz_b200/parallel.py).
"ddh" block  (BASELINE configs[2]/[3], every N): the 2048^2, n_basis 4, omega 100, block-16 DDH operator (262 144 subdomains)
    STRONG-scaled over the N ranks through the library's distributed DDH (subdomain slabs, traces packed in the kernel epilogue,
    ncclSend/ncclRecv, masked inner products + ncclAllReduce): action time, FP32 TFLOP/s against the non-tensor FP32 peak, bytes
    exchanged, a time-boxed GMRES(30) restart cycle, and the convergent 512^2 solve of the examples/DDH.cpp flow (restart count
    must not depend on N).
`--impl reference` times the CPU restatement of the reference's kernels (oracle/, OpenMP over all host cores; the reference
has no host-only build, SURVEY R6) on the SAME 1024^2 workload, index data from the oracle's own closed-form numpy setup (the
product library is not loaded). Prints ONE JSON line on rank 0.
`--dump-outputs DIR` writes y = A [u; v] of the last timed step to DIR (see dump_outputs), so that two builds can be compared
output for output: the inputs depend on nothing but the arguments.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "helmholtz_operator_apply_gdofs"
UNIT = "GDOF/s"
DUMP_VALUES = 1 << 22  # --dump-outputs: float64 entries of y written at most, over all ranks (32 MiB)


def coef(x, y):
    return 1.0 + 0.5 * np.sin(np.pi * x) * np.cos(np.pi * y)


def dump_sample(n, world):
    """positions kept by --dump-outputs in a vector of n entries: all of them when n fits this rank's share of DUMP_VALUES,
    else one entry drawn from each of that many equal strata with a fixed seed (a function of n and world only)"""
    k = DUMP_VALUES // world
    if n <= k:
        return np.arange(n, dtype=np.int64)
    edges = np.arange(k + 1, dtype=np.int64) * n // k
    return edges[:-1] + np.random.default_rng(2024).integers(0, np.diff(edges))


def dump_outputs(out_dir, take, n, rank, world):
    """y = A [u; v] as the caller of the timed apply receives it, as DIR/helmholtz_y.npy (float64): the entries dump_sample(n, world)
    picks, in increasing position. take(idx) returns y[idx] as a numpy array. N > 1: one file per rank (helmholtz_y_rank<r>.npy),
    DUMP_VALUES entries in all."""
    idx = dump_sample(n, world)
    name = "helmholtz_y%s.npy" % ("_rank%d" % rank if world > 1 else "")
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name), np.asarray(take(idx), np.float64))
    return {"dir": out_dir, "file": name, "entries": len(idx), "of": n,
            "positions": "bench.dump_sample(%d, %d): one entry per stratum, seed 2024" % (n, world) if len(idx) < n else "all"}


def workload(args):
    return ("Helmholtz composite apply (stiffness + weighted mass on u and v + boundary face mass), uniform_rect(%d x %d) per GPU, "
            "n_basis %d (degree %d), omega %g" % (args.nx, args.nx, args.nb, args.nb - 1, args.omega))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons during the timed regions (B200_PROFILING.md recipe). NVML in-process (a query takes
    microseconds, so even a 20 ms region gets several samples); falls back to polling nvidia-smi."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index, period=0.002):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.period = index, [], False, period
        self.nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # LOCAL_RANK indexes the visible devices: map through CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis and all(v.strip().isdigit() for v in vis.split(",")):
                phys = int(vis.split(",")[index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nv = pynvml
        except Exception:
            self.nv = None

    def _nvml_row(self):
        nv = self.nv
        sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
        mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
            else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        bit = lambda name: "Active" if (r & getattr(nv, name, 0)) else "Not Active"
        return [str(sm), str(mx), bit("nvmlClocksThrottleReasonHwSlowdown"), bit("nvmlClocksThrottleReasonHwThermalSlowdown"),
                bit("nvmlClocksThrottleReasonSwThermalSlowdown"), bit("nvmlClocksThrottleReasonSwPowerCap")]

    def run(self):
        while not self.stop_flag and self.nv is not None:
            try:
                self.rows.append(self._nvml_row())
            except Exception:
                self.nv = None
                break
            time.sleep(self.period)
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows), "source": "nvml" if self.nv is not None else "nvidia-smi"}


# ---- CPU restatement of the reference's kernels on the SAME workload (oracle only: the product library is not touched) ----
def cpu_port_setup(nx, nb, omega):
    from oracle import ops as O
    from oracle import setup_np as S
    c = S.uniform_rect_closed_form(nx, -1.0, 1.0, nx, -1.0, 1.0, S.Basis(nb))
    ofem = O.H1.from_arrays(nb, c["I"], c["xy"], c["corners"])
    ofs = O.FaceSpace.from_arrays(ofem, c["face_I"], c["face_proj"], c["face_meas"])
    a = coef(c["xy"][:, 0], c["xy"][:, 1])
    return O.Helmholtz(omega, a * a, a[ofs.proj], ofem, ofs), ofem.ndof


def time_cpu_port(nx, nb, omega, steps, warmup):
    from oracle import ops as O
    O.set_threads(os.cpu_count() or 1)  # all host threads, whatever OMP_NUM_THREADS the launcher exported
    A, ndof = cpu_port_setup(nx, nb, omega)
    x = np.random.default_rng(12345).uniform(-1, 1, 2 * ndof)
    for _ in range(warmup):
        A.action(x)
    t0 = time.perf_counter()
    for _ in range(steps):
        y = A.action(x)
    dt = (time.perf_counter() - t0) / steps
    return 2 * ndof / dt / 1e9, dt, O.max_threads(), ndof, y


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    val, dt, cores, ndof, y = time_cpu_port(args.nx, args.nb, args.omega, args.steps, args.warmup)
    sample = "the full uniform_rect(%d) n_basis %d workload (one slab), %d applies of %.3f s, OpenMP %d threads" % (
        args.nx, args.nb, args.steps, dt, cores)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload(args), "ndof_per_gpu": ndof, "parallelism": "slab%d" % args.gpus},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "the reference has no host-only build (all operator bodies are __device__ lambdas, SURVEY R6); this arm is the CPU "
                    "restatement in oracle/oracle.c on one 1024^2 slab (one CPU run whatever N is), index data from "
                    "oracle/setup_np.py:uniform_rect_closed_form (pinned to the reference's own 1024^2 hashes); libcuddh_b200.so is not loaded"}
    if args.dump_outputs:  # same x as rank 0 of the GPU path, same positions: comparable file for file with a single-GPU dump
        line["dump_outputs"] = dump_outputs(args.dump_outputs, lambda idx: y[idx], y.size, 0, 1)
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed applies of the headline (device-resident) loop; the end-to-end leg runs "
                    "max(6, min(steps, 12)) requests and the roofline kernel timing max(steps, 20) launches")
    ap.add_argument("--warmup", type=int, default=3, help="untimed applies before the timed loop (at least 3)")
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--nx", type=int, default=1024)
    ap.add_argument("--nb", type=int, default=5)
    ap.add_argument("--omega", type=float, default=100.0)
    ap.add_argument("--no-extras", action="store_true", help="skip the context numbers (reference GPU kernels, n_basis 4, Krylov kernels)")
    ap.add_argument("--no-ddh", action="store_true", help="skip the DDH block (config 3 action / cycle and the 512^2 solve)")
    ap.add_argument("--ddh-nx", type=int, default=2048)
    ap.add_argument("--ddh-solve-nx", type=int, default=512)
    ap.add_argument("--ddh-ho-nx", type=int, default=512, help="mesh of the scaled-down high-order (configs[4]) DDH action")
    ap.add_argument("--ddh-box-seconds", type=float, default=45.0, help="time box of the GMRES(30) restart cycle at config 3")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write y = A [u; v] of the last timed step to DIR/*.npy (a fixed, seeded sample of at most %d entries over all ranks)" % DUMP_VALUES)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist
    import cuddhelmholtz_b200 as cb
    from cuddhelmholtz_b200.parallel import GpuSlabHelmholtz

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback for the product path)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    cb.load()
    comm = cb.Comm(rank, world) if world > 1 else None  # the library's own NCCL communicator (id broadcast through torch.distributed)

    nx, nb, omega, K, W = args.nx, args.nb, args.omega, args.steps, args.warmup
    slab = GpuSlabHelmholtz(nx, nx, nb, omega, coef, rank, world, comm=comm)
    ndof = slab.ndof
    hx = torch.from_numpy(np.random.default_rng(12345 + rank).uniform(-1, 1, 2 * ndof)).pin_memory()
    hy = torch.empty(2 * ndof, dtype=torch.float64).pin_memory()
    x = hx.cuda()
    y = torch.empty_like(x)
    if world > 1:  # make x consistent on the interface rows (both neighbours must hold the same values)
        slab.exchange(x)
        x.mul_(1.0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident timing ----
    for _ in range(W):
        slab.apply(x, y)
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    l0 = cb.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(K):
        slab.apply(x, y)
    e1.record()
    barrier()
    launches = cb.launch_count() - l0
    ms_step = max_over_ranks(e0.elapsed_time(e1)) / K
    value = 2.0 * ndof * world / (ms_step * 1e-3) / 1e9
    # y still holds the last timed step's result (the legs below overwrite it)
    dumped = None
    if args.dump_outputs:
        dumped = dump_outputs(args.dump_outputs, lambda idx: y[torch.as_tensor(idx, device=y.device)].cpu().numpy(), y.numel(), rank, world)

    # ---- end to end through the public API with HOST buffers: every step copies its [u; v] from pinned host memory, applies
    # the operator and reads the result back to the host. Consecutive steps are independent requests, so they are
    # kept in flight on three streams with their own buffers: the H2D of step k+1 overlaps the apply / D2H of step k (PCIe is full duplex). ----
    Ke = max(6, min(K, 12))
    NS = 3  # requests in flight
    streams = [torch.cuda.Stream() for _ in range(NS)]
    xb, yb = [x] + [torch.empty_like(x) for _ in range(NS - 1)], [y] + [torch.empty_like(y) for _ in range(NS - 1)]
    hyb = [hy] + [torch.empty(2 * ndof, dtype=torch.float64).pin_memory() for _ in range(NS - 1)]

    lanes = [slab.lane(b) for b in range(NS)]  # one exchange handle per stream in flight (N > 1); lane 0 = the slab itself

    def e2e_steps(n):
        for k in range(n):
            b = k % NS
            with torch.cuda.stream(streams[b]):
                xb[b].copy_(hx, non_blocking=True)
                lanes[b].apply(xb[b], yb[b])
                hyb[b].copy_(yb[b], non_blocking=True)

    for st in streams:
        st.wait_stream(torch.cuda.current_stream())
    e2e_steps(NS)
    barrier()
    e0.record()
    for st in streams:
        st.wait_event(e0)
    e2e_steps(Ke)
    for st in streams:
        torch.cuda.current_stream().wait_stream(st)
    e1.record()
    barrier()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1)) / Ke
    e2e_value = 2.0 * ndof * world / (e2e_ms * 1e-3) / 1e9
    # the same without overlap (one stream, copy -> apply -> copy per step), for reference
    barrier()
    e0.record()
    for _ in range(3):
        x.copy_(hx, non_blocking=True)
        slab.apply(x, y)
        hy.copy_(y, non_blocking=True)
    e1.record()
    barrier()
    e2e_serial_ms = e0.elapsed_time(e1) / 3
    if sampler:  # clocks are sampled across both timed regions (device-resident and end-to-end)
        sampler.stop_flag = True
    del xb, yb, hyb, lanes
    torch.cuda.empty_cache()

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload(args), "ndof_per_gpu": ndof, "parallelism": "slab%d" % world,
                       "l2": "inputs larger than L2 (x,y 2x%.0f MB, metric data %.0f MB)" % (
                           16 * ndof / 1e6, (24 * (nb + 1) ** 2 + 8 * (1 + 3 * nb // 2 + 1) ** 2) * nx * nx / 1e6)},
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms, "h2d_bytes_per_step": 16 * ndof, "d2h_bytes_per_step": 16 * ndof,
                    "steps": Ke, "pipelining": "three streams / buffer sets in flight: H2D of step k+1 overlaps apply + D2H of step k",
                    "ms_per_step_unpipelined": e2e_serial_ms,
                    "note": None if world == 1 else "all ranks stream through the same host memory / PCIe root complex: this leg measures the "
                                                    "host link of the box, not the kernels (see ms_per_step for the device-resident number)"},
            "gpu_launches": int(launches), "clocks": sampler.summary() if sampler else None}
    if world > 1:
        line["exchange"] = slab.exchange_info()
    if dumped:
        line["dump_outputs"] = dumped

    # ---- roofline of the dominant kernel, timed alone with CUDA events on its stream: the fused Helmholtz volume kernel
    # (S - omega^2 M on u and v; > 90 % of the step). Algorithmic bytes = SURVEY §8(d) fused formulation per element. ----
    if rank == 0:
        line["roofline"], line["operators"] = roofline_block(cb, torch, slab, x, y, nb, nx, ndof, ms_step, K)
    barrier()

    # ---- DDH-GMRES (path B) on the N ranks ----
    if not args.no_ddh:
        try:
            d = ddh_block(args, cb, torch, dist, comm, rank, world, local_rank)
        except Exception as e:  # keep the headline if the big case cannot run (e.g. out of host memory on a small box)
            d = "failed: %r" % (e,)
        if rank == 0:
            line["ddh"] = d
            if isinstance(d, dict) and "roofline_fp32" in d:
                line["roofline"]["fp32_ddh_action"] = d["roofline_fp32"]

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- CPU baseline: the oracle port on the box's host cores, bounded sample of the same workload ----
    if world == 1:
        try:
            val, dt, cores, nd, _ = time_cpu_port(nx, nb, omega, 3, 1)
            line["cpu_baseline"] = {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": "the full uniform_rect(%d) n_basis %d workload, 3 applies of %.2f s (+1 warm-up)" % (nx, nb, dt)}
        except Exception as e:  # the checker is optional for the number, never for the product
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %r" % (e,)}
        if not args.no_extras:
            line["context"] = extras(args, cb, torch, slab, x, y)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def roofline_block(cb, torch, slab, x, y, nb, nx, ndof, ms_step, K):
    """roofline of the dominant kernel (the fused Helmholtz volume kernel; > 90 % of the step), timed alone with CUDA events on its
    stream. `achieved` / `frac` use the ALGORITHMIC bytes of SURVEY §8(d) (the reference's stored-metric formulation: 24 nq_S^2 + 8
    nq_M^2 + 4 nb^2 + 32 (nb-1)^2 per element). On a uniform (all-affine) mesh the library runs the stiffness phase from three
    per-element constants instead of the stored metric, so fewer bytes actually move: `moved` carries the roofline of THAT
    formulation, and `stored_metric` the same measurement with the stored-metric kernel (CUDDH_B200_AFFINE=0) - both rooflines."""
    peak, peak_src = measured_peaks()
    nqs, nqm = nb + 1, 1 + 3 * nb // 2 + 1
    u, yy = x[:ndof], y[:ndof]
    reps = max(K, 20)

    def measure(op, xa, ya, step_ms=None):
        # the dominant kernel cannot take longer than the step it is part of: re-measure (clock ramp) if it seems to
        for attempt in range(3):
            ms_patch, ms_rest = op.time_phases(xa, ya, reps)
            if step_ms is None or ms_patch + ms_rest <= 1.02 * step_ms:
                break
        return ms_patch, ms_rest

    fused = slab.op.is_fused()
    if fused:
        op, xa, ya = slab.op, x, y
        kname = "volume_action_ws<%d,%d,stiffness,%d%s> (fused S - w^2 M on [u;v])" % (nb, nqs, nqm, ",affine" if op.is_affine() else "")
        tkey = "helmholtz%s_%d_%d_%d_nx%d" % ("_affine" if op.is_affine() else "", nb, nqs, nqm, nx)
    else:
        op, xa, ya = cb.StiffnessMatrix(slab.fem), u, yy
        kname, tkey = "volume_action_kernel<%d,%d,stiffness>" % (nb, nqs), "stiffness_%d_%d_nx%d" % (nb, nqs, nx)
    ms_patch, ms_rest = measure(op, xa, ya, ms_step if fused else None)
    bytes_k, bytes_m = op.algorithmic_bytes(), op.moved_bytes()
    roof = {"bound": "hbm", "kernel": kname, "achieved": bytes_k / (ms_patch * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
            "peak_source": peak_src, "ms_per_launch": ms_patch, "algorithmic_bytes": bytes_k, "rest_of_step_ms": ms_rest,
            "timing": "median of %d launches after 3 warm applies, CUDA events on the launch stream" % reps,
            "consistent_with_step": bool(not fused or ms_patch + ms_rest <= 1.02 * ms_step), "traffic": None,
            "formulation": ("stiffness metric from 3 per-element constants (all elements affine), mass metric stored" if op.is_affine()
                            else "stored metric (the reference's formulation)")}
    roof["frac"] = roof["achieved"] / peak
    roof["moved"] = {"bytes": bytes_m, "achieved": bytes_m / (ms_patch * 1e-3) / 1e9, "frac": bytes_m / (ms_patch * 1e-3) / 1e9 / peak,
                     "note": "algorithmic bytes of the formulation this kernel runs (equal to algorithmic_bytes unless affine)"}
    flops = float(nx) * nx * 2 * (8 * nqs * nb * (nb + nqs) + 6 * nqs * nqs + 4 * nqm * nb * (nb + nqm) + nqm * nqm)
    roof["fp64"] = {"flops": flops, "achieved_tflops": flops / (ms_patch * 1e-3) / 1e12,
                    "note": "SURVEY §8(a) flop counts of S and M on both fields; the B200 FP64 FMA pipe issues one warp DFMA per 2 cycles per "
                            "SM sub-partition (~37 TFLOP/s at 1965 MHz), see profiles/r02_notes.md for the ncu pipe utilisation"}
    tr = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tr):
        try:
            roof["traffic"] = json.load(open(tr)).get(tkey)
        except Exception:
            pass
    if fused and op.is_affine():  # the other roofline: the stored-metric kernel on the same data
        os.environ["CUDDH_B200_AFFINE"] = "0"
        try:
            gen = cb.Helmholtz(slab.op.omega, slab._a2, slab._af, slab.fem, slab.fs_phys)
            assert not gen.is_affine()
            yg = torch.empty_like(y)
            gen.action(x, yg)
            gp, gr = measure(gen, x, yg)
            agree = float((yg - y).norm() / y.norm()) if slab.world == 1 else None  # y holds the last apply of the same x (N = 1)
            gb = gen.algorithmic_bytes()
            roof["stored_metric"] = {"kernel": "volume_action_ws<%d,%d,stiffness,%d> (CUDDH_B200_AFFINE=0)" % (nb, nqs, nqm), "ms_per_launch": gp,
                                     "rest_of_step_ms": gr, "achieved": gb / (gp * 1e-3) / 1e9, "frac": gb / (gp * 1e-3) / 1e9 / peak,
                                     "rel_diff_vs_affine_result": agree}
            try:
                roof["stored_metric"]["traffic"] = json.load(open(tr)).get("helmholtz_%d_%d_%d_nx%d" % (nb, nqs, nqm, nx))
            except Exception:
                pass
            del gen, yg
        except Exception as e:
            roof["stored_metric"] = "failed: %r" % (e,)
        finally:
            del os.environ["CUDDH_B200_AFFINE"]
        torch.cuda.empty_cache()
    Sop = cb.StiffnessMatrix(slab.fem)
    sp_, ss_ = Sop.time_phases(u, yy, reps)
    Mop = cb.MassMatrix(slab._a2, slab.fem)
    mp_, ms_ = Mop.time_phases(u, yy, reps)
    per_op = {"stiffness": {"ms": sp_ + ss_, "gdofs": ndof / ((sp_ + ss_) * 1e-3) / 1e9, "kernel_ms": sp_, "affine": Sop.is_affine(),
                            "hbm_frac_kernel": Sop.algorithmic_bytes() / (sp_ * 1e-3) / 1e9 / peak,
                            "hbm_frac_kernel_moved_bytes": Sop.moved_bytes() / (sp_ * 1e-3) / 1e9 / peak},
              "mass_weighted": {"ms": mp_ + ms_, "gdofs": ndof / ((mp_ + ms_) * 1e-3) / 1e9, "kernel_ms": mp_,
                                "hbm_frac_kernel": Mop.algorithmic_bytes() / (mp_ * 1e-3) / 1e9 / peak},
              "helmholtz_composite": {"ms": ms_step, "hbm_frac_fused_formulation": slab.op.algorithmic_bytes() / (ms_step * 1e-3) / 1e9 / peak}}
    del Mop, Sop
    torch.cuda.empty_cache()
    return roof, per_op


def ddh_problem(cb, torch, nx, nb, omega):
    """mesh, space, coefficient and load vector of examples/DDH.cpp:61-123 at a chosen size"""
    mesh = cb.Mesh2D.uniform_rect(nx, -1.0, 1.0, nx, -1.0, 1.0)
    fem = cb.H1Space(mesh, cb.Basis(nb))
    xy = fem.physical_coordinates()
    X, Y = xy[:, 0], xy[:, 1]
    ha = np.where(X * X + Y * Y < 0.0625, 0.2, 1.0)
    s = omega * omega
    src = s / np.pi * np.exp(-s * ((X + 0.5) ** 2 + Y ** 2)) + s / np.pi * np.exp(-s * ((X - 0.5) ** 2 + (Y + 0.5) ** 2))
    n = fem.size()
    f = torch.zeros(2 * n, dtype=torch.float64, device="cuda")
    M = cb.MassMatrix(fem)
    M.action(torch.as_tensor(src, device="cuda"), f[:n])
    del M
    return mesh, fem, ha, f, n


def fp32_peak_tflops(torch, sm_max_mhz):
    # non-tensor FP32: 128 FMA lanes per SM per clock
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return sms * 128 * 2 * (sm_max_mhz or 1965.0) * 1e6 / 1e12


def ddh_block(args, cb, torch, dist, comm, rank, world, local_rank):
    """BASELINE configs[2]/[3]: the config-3 operator strong-scaled over the ranks (same problem at every N), then the convergent
    512^2 solve. All timings are CUDA events on the launch stream, max over ranks."""
    out = {"n_gpus": world, "scaling": "strong (same 2048^2 problem at every N)"}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def tmax(v):
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    ev = lambda: torch.cuda.Event(enable_timing=True)
    # ---------------- config 3: uniform_rect(2048), n_basis 4, omega 100, block 16 ----------------
    nx, nb, omega = args.ddh_nx, 4, 100.0
    t0 = time.perf_counter()
    mesh, fem, ha, f, n = ddh_problem(cb, torch, nx, nb, omega)
    D = cb.DDH(omega, ha, fem, nx, nx, 16)
    A = cb.DDHDist(D, comm, rank, world)
    setup_s = time.perf_counter() - t0
    info, di = D.info(), A.info()
    m = D.size()
    b = torch.empty(m, dtype=torch.float32, device="cuda")
    y = torch.empty(m, dtype=torch.float32, device="cuda")
    sampler = ClockSampler(local_rank, period=0.05) if rank == 0 else None
    if sampler:
        sampler.start()
    barrier()
    e0, e1, e2 = ev(), ev(), ev()
    e0.record()
    A.rhs(f, b)           # also the warm-up of the kernel
    e1.record()
    A.action(b, y)
    e2.record()
    barrier()
    rhs_ms, act_ms = tmax(e0.elapsed_time(e1)), tmax(e1.elapsed_time(e2))
    flops = D.flops()
    peak = None
    c3 = {"nx": nx, "n_basis": nb, "omega": omega, "block": 16, "n_domains": info["n_domains"], "nt": info["nt"], "n_lambda": m,
          "kernel_kind": D.kernel_kind(), "host_setup_s": setup_s, "rhs_ms": rhs_ms, "action_ms": act_ms,
          "action_fp32_tflops": flops / (act_ms * 1e-3) / 1e12, "subdomains_this_rank": di["dom_end"] - di["dom_begin"],
          "exchange_bytes_per_action_rank0": di["bytes_per_action"], "neighbours_rank0": di["n_peers"]}
    # one time-boxed GMRES(m) restart cycle (m <= 30 chosen so that the cycle fits the box: ~m + 2 actions)
    mbox = int(max(2, min(30, args.ddh_box_seconds / max(act_ms * 1e-3, 1e-6) - 2)))
    L = torch.zeros(m, dtype=torch.float32, device="cuda")
    barrier()
    e0.record()
    res = A.solve(b, L, m=mbox, maxit=2, tol=1e-4, orth=cb.CGS2)
    e1.record()
    barrier()
    cyc_ms = tmax(e0.elapsed_time(e1))
    if sampler:
        sampler.stop_flag = True
        clk = sampler.summary()
        peak = fp32_peak_tflops(torch, clk.get("sm_max_mhz"))
        c3["clocks"] = clk
    c3["gmres_cycle"] = {"m": mbox, "m_target": 30, "time_box_s": args.ddh_box_seconds, "seconds": cyc_ms / 1e3, "matvecs": res.num_matvec,
                         "rel_residual_before": 1.0, "rel_residual_after": (res.res_norm[-1] / res.res_norm[0]) if res.res_norm and res.res_norm[0] > 0 else None,
                         "allreduces": res.allreduces, "reorthogonalisations": res.reorth,
                         "note": "x0 = 0, so the residual before the cycle is ||b||; 1024^2 and larger do not converge within maxit 100 "
                                 "restarts in the reference's algorithm either (no coarse space; profiles/r01_ddh_ladder.jsonl)"}
    out["config3"] = c3
    if peak:
        out["roofline_fp32"] = {"bound": "fp32 (non-tensor FMA issue; HBM idle: ~7 KB read per subdomain per action)", "kernel": "ddh_kernel_reg4",
                                "achieved": c3["action_fp32_tflops"], "peak": peak, "unit": "TFLOP/s", "frac": c3["action_fp32_tflops"] / peak,
                                "peak_source": "SMs x 128 lanes x 2 x max SM clock (NVML)", "n_gpus": world,
                                "flops": "the reference's count n_domains*5*nt*256*(2(8nb+7)+26) (BASELINE.md §3)"}
        if world > 1:
            out["roofline_fp32"]["peak"] = peak * world
            out["roofline_fp32"]["frac"] = c3["action_fp32_tflops"] / (peak * world)
    del A, D, b, y, L, f, fem, mesh
    torch.cuda.empty_cache()

    # ---------------- BASELINE configs[4] order, scaled to 1/16 of its subdomains: n_basis 8, block 32, same nt ----------------
    try:
        nx5, omega5 = args.ddh_ho_nx, 400.0 * args.ddh_ho_nx / 2048.0
        mesh, fem, ha, f, n = ddh_problem(cb, torch, nx5, 8, omega5)
        D = cb.DDH(omega5, ha, fem, nx5, nx5, 32)
        A = cb.DDHDist(D, comm, rank, world)
        m5 = D.size()
        b = torch.empty(m5, dtype=torch.float32, device="cuda")
        y = torch.empty(m5, dtype=torch.float32, device="cuda")
        barrier()
        e0, e1, e2 = ev(), ev(), ev()
        e0.record()
        A.rhs(f, b)
        e1.record()
        A.action(b, y)
        e2.record()
        barrier()
        a5 = tmax(e1.elapsed_time(e2))
        out["config5_scaled"] = {"nx": nx5, "n_basis": 8, "omega": omega5, "block": 32, "n_domains": D.info()["n_domains"], "nt": D.info()["nt"],
                                 "n_lambda": m5, "kernel_kind": D.kernel_kind(), "rhs_ms": tmax(e0.elapsed_time(e1)), "action_ms": a5,
                                 "action_fp32_tflops": D.flops() / (a5 * 1e-3) / 1e12,
                                 "note": "configs[4] (2048^2, omega 400, block 32) has 16x the subdomains and the same nt; its action scales "
                                         "linearly in the subdomain count (%.1f s on this many GPUs by this measurement)" % (16 * a5 / 1e3)}
        del A, D, b, y, f, fem, mesh
        torch.cuda.empty_cache()
    except Exception as e:
        out["config5_scaled"] = "failed: %r" % (e,)

    # ---------------- the convergent solve: examples/DDH.cpp flow at 512^2 (omega = 2 pi nx / 10, GMRES(20), tol 1e-4) ----------------
    nx = args.ddh_solve_nx
    omega = 2 * np.pi * nx / 10
    mesh, fem, ha, f, n = ddh_problem(cb, torch, nx, nb, omega)
    D = cb.DDH(omega, ha, fem, nx, nx, 16)
    A = cb.DDHDist(D, comm, rank, world)
    m = D.size()
    b = torch.empty(m, dtype=torch.float32, device="cuda")
    L = torch.zeros(m, dtype=torch.float32, device="cuda")
    A.rhs(f, b)
    barrier()
    e0.record()
    res = A.solve(b, L, m=20, maxit=100, tol=1e-4)   # library default orthogonalisation (MGS: the reference's arithmetic)
    e1.record()
    U = torch.empty(2 * n, dtype=torch.float64, device="cuda")
    A.postprocess(L, f, U)
    e2.record()
    barrier()
    out["solve"] = {"nx": nx, "n_basis": nb, "omega": omega, "n_domains": D.info()["n_domains"], "nt": D.info()["nt"], "n_lambda": m,
                    "gmres_m": 20, "tol": 1e-4, "seconds": tmax(e0.elapsed_time(e1)) / 1e3, "postprocess_ms": tmax(e1.elapsed_time(e2)),
                    "restarts": res.num_iter, "matvecs": res.num_matvec, "success": res.success, "allreduces": res.allreduces,
                    "solution_norm": float(U.norm()),
                    "reference_library_same_gpu": "92 restarts / 1888 matvecs in 419.9 s on one B200 (profiles/r01_ddh_ladder.jsonl)" if nx == 512 else None}
    return out


def extras(args, cb, torch, slab, x, y):
    """context numbers next to the headline (N = 1 only): the reference's own CUDA kernels (sm_100 build of the unmodified
    sources) on this GPU, the other order (n_basis 4), the Krylov kernels, and the examples' solves against the reference library."""
    out = {}
    peak, _ = measured_peaks()
    drv = os.path.join(ROOT, "oracle", "_ref", "ref_driver")
    if os.path.exists(drv):
        try:
            r = subprocess.run([drv, "time_ops", str(args.nx), str(args.nb), str(args.omega), "10"], capture_output=True, text=True, timeout=600)
            out["reference_gpu_kernels"] = json.loads(r.stdout.strip().splitlines()[-1])
        except Exception as e:
            out["reference_gpu_kernels"] = "failed: %r" % (e,)
    try:  # Krylov vector kernels at the headline size: one GMRES(30) restart cycle on the Helmholtz composite, both orthogonalisations
        n2 = x.numel()
        bb = torch.rand(n2, dtype=torch.float64, device="cuda") - 0.5
        kk = {}
        for name, mode in (("mgs", cb.MGS), ("cgs2", cb.CGS2)):
            xx = torch.zeros(n2, dtype=torch.float64, device="cuda")
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            o = cb.gmres(n2, xx, slab.op, bb, 30, 2, 1e-12, orth=mode, time_orth=True)
            torch.cuda.synchronize()
            kk[name] = {"cycle_seconds": time.perf_counter() - t0, "matvecs": o.num_matvec, "orth_ms": o.orth_ms, "orth_gbytes": o.orth_bytes / 1e9,
                        "orth_gbs": o.orth_bytes / max(o.orth_ms, 1e-9) / 1e6, "hbm_frac": o.orth_bytes / max(o.orth_ms, 1e-9) / 1e6 / peak,
                        "reorth": o.reorth, "rel_residual": o.res_norm[-1] / o.res_norm[0]}
            del xx
        out["gmres_vector_kernels"] = dict(kk, n=n2, m=30, note="orth_* = Gram-Schmidt kernels only (CUDA events), bytes = vectors read + written")
        del bb
        torch.cuda.empty_cache()
    except Exception as e:
        out["gmres_vector_kernels"] = "failed: %r" % (e,)
    try:  # the other reading of "p=4" (SURVEY R3): n_basis 4 (degree 3), the order the DDH configs use
        mesh = cb.Mesh2D.uniform_rect(args.nx, -1.0, 1.0, args.nx, -1.0, 1.0)
        fem = cb.H1Space(mesh, cb.Basis(4))
        n4 = fem.size()
        xx = torch.rand(n4, dtype=torch.float64, device="cuda") - 0.5
        yy = torch.empty_like(xx)
        aa = torch.rand(n4, dtype=torch.float64, device="cuda") + 0.5
        res = {"ndof": n4}
        for name, op in (("stiffness", cb.StiffnessMatrix(fem)), ("mass_weighted", cb.MassMatrix(aa, fem))):
            op.action(xx, yy)
            pms, sms = op.time_phases(xx, yy, 20)
            res[name] = {"ms": pms + sms, "gdofs": n4 / ((pms + sms) * 1e-3) / 1e9, "hbm_frac_patch_kernel": op.algorithmic_bytes() / (pms * 1e-3) / 1e9 / peak}
        try:  # the fused Helmholtz composite at this order (own try: the numbers above survive a failure here)
            fs4 = cb.FaceSpace(fem, mesh.boundary_edges())
            af = torch.ones(fs4.size(), dtype=torch.float64, device="cuda")
            H4 = cb.Helmholtz(args.omega, aa, af, fem, fs4)
            x2 = torch.rand(2 * n4, dtype=torch.float64, device="cuda") - 0.5
            y2 = torch.empty_like(x2)
            H4.action(x2, y2)
            pms, rest = H4.time_phases(x2, y2, 20)
            res["helmholtz_composite"] = {"ms": pms + rest, "gdofs": 2 * n4 / ((pms + rest) * 1e-3) / 1e9, "kernel_ms": pms,
                                          "hbm_frac_kernel": H4.algorithmic_bytes() / (pms * 1e-3) / 1e9 / peak, "kernel_kind": H4.kernel_kind()}
            del H4, fs4, af, x2, y2
        except Exception as e:
            res["helmholtz_composite"] = "failed: %r" % (e,)
        out["n_basis_4"] = res
        del mesh, fem, xx, yy, aa
        torch.cuda.empty_cache()
    except Exception as e:
        out["n_basis_4"] = "failed: %r" % (e,)
    try:  # high order (BASELINE configs[4]): n_basis 8 operators at 1024^2
        out["n_basis_8"] = high_order_ops(cb, torch, args.nx, 8, peak)
    except Exception as e:
        out["n_basis_8"] = "failed: %r" % (e,)
    try:
        out["n_basis_9"] = high_order_ops(cb, torch, args.nx, 9, peak)
    except Exception as e:
        out["n_basis_9"] = "failed: %r" % (e,)
    try:  # BASELINE configs[4] order on one GPU: n_basis 8 DDH action, the reference's block 16 and the config's block 32
        out["ddh_n_basis_8"] = ddh_high_order(cb, torch, drv if os.path.exists(drv) else None)
    except Exception as e:
        out["ddh_n_basis_8"] = "failed: %r" % (e,)
    try:
        out["ddh_example_128"] = ddh_example(cb, torch, drv if os.path.exists(drv) else None)
    except Exception as e:
        out["ddh_example_128"] = "failed: %r" % (e,)
    try:
        out["helmholtz_example_128"] = helmholtz_example(cb, torch, drv if os.path.exists(drv) else None)
    except Exception as e:
        out["helmholtz_example_128"] = "failed: %r" % (e,)
    return out


def high_order_ops(cb, torch, nx, nb, peak):
    mesh = cb.Mesh2D.uniform_rect(nx, -1.0, 1.0, nx, -1.0, 1.0)
    fem = cb.H1Space(mesh, cb.Basis(nb))
    n = fem.size()
    xx = torch.rand(n, dtype=torch.float64, device="cuda") - 0.5
    yy = torch.empty_like(xx)
    aa = torch.rand(n, dtype=torch.float64, device="cuda") + 0.5
    res = {"ndof": n, "nx": nx, "kernel": "volume_action_pair (thread pair per element, kernel_kind 3)",
           "hbm_frac_patch_kernel": "SURVEY 8(d) bytes of the reference's stored-metric formulation / patch-kernel time / measured HBM peak"}

    def one(mk):
        op = mk()
        op.action(xx, yy)
        pms, sms = op.time_phases(xx, yy, 10)
        r = {"ms": pms + sms, "kernel_ms": pms, "gdofs": n / ((pms + sms) * 1e-3) / 1e9, "kernel_kind": op.kernel_kind(),
             "affine": op.is_affine(), "hbm_frac_patch_kernel": op.algorithmic_bytes() / (pms * 1e-3) / 1e9 / peak}
        del op
        torch.cuda.empty_cache()
        return r

    res["stiffness"] = one(lambda: cb.StiffnessMatrix(fem))
    if res["stiffness"]["affine"] and "CUDDH_B200_AFFINE" not in os.environ:  # the stored-metric instance on the same data
        os.environ["CUDDH_B200_AFFINE"] = "0"
        try:
            res["stiffness_stored_metric"] = one(lambda: cb.StiffnessMatrix(fem))
        finally:
            del os.environ["CUDDH_B200_AFFINE"]
    res["mass_weighted"] = one(lambda: cb.MassMatrix(aa, fem))
    # the Helmholtz composite at this order: n_basis 6-8 on affine meshes run both phases of a field in one launch of the thread-pair kernel
    fs = cb.FaceSpace(fem, mesh.boundary_edges())
    af = torch.ones(fs.size(), dtype=torch.float64, device="cuda")
    x2 = torch.rand(2 * n, dtype=torch.float64, device="cuda") - 0.5
    y2 = torch.empty_like(x2)
    H = cb.Helmholtz(100.0, aa, af, fem, fs)
    H.action(x2, y2)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        H.action(x2, y2)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    res["helmholtz_composite"] = {"ms": ms, "gdofs": 2 * n / (ms * 1e-3) / 1e9, "kernel_kind": H.kernel_kind(),
                                  "hbm_frac_reference_formulation": H.algorithmic_bytes() / (ms * 1e-3) / 1e9 / peak}
    del H
    torch.cuda.empty_cache()
    return res


def ddh_high_order(cb, torch, drv, nx=128, nb=8):
    """one DDH action at n_basis 8 (generic one-thread-per-node kernel: no register-tiled variant for this order yet)"""
    omega = 2 * np.pi * nx / 10
    mesh = cb.Mesh2D.uniform_rect(nx, -1.0, 1.0, nx, -1.0, 1.0)
    fem = cb.H1Space(mesh, cb.Basis(nb))
    res = {"nx": nx, "n_basis": nb, "omega": omega}
    for block in (16, 32):
        D = cb.DDH(omega, np.ones(fem.size()), fem, nx, nx, block)
        m = D.size()
        x = torch.rand(m, dtype=torch.float32, device="cuda")
        y = torch.empty_like(x)
        D.action(x, y)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        D.action(x, y)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        res["block_%d" % block] = {"n_domains": D.info()["n_domains"], "nt": D.info()["nt"], "action_ms": ms, "kernel_kind": D.kernel_kind(),
                                   "action_fp32_tflops": D.flops() / (ms * 1e-3) / 1e12}
        del D, x, y
    if drv:
        try:
            r = subprocess.run([drv, "time_ddh", str(nx), str(nb), repr(float(omega)), "1"], capture_output=True, text=True, timeout=900)
            res["reference_gpu_kernel_block_16"] = json.loads(r.stdout.strip().splitlines()[-1])
        except Exception as e:
            res["reference_gpu_kernel_block_16"] = "failed: %r" % (e,)
    return res


def ddh_example(cb, torch, drv, nx=128, nb=4):
    """examples/DDH.cpp: uniform_rect(128), n_basis 4, omega = 2 pi 12.8, FP32 GMRES(20), maxit 100, tol 1e-4."""
    omega = 2 * np.pi * nx / 10
    mesh, fem, ha, f, n = ddh_problem(cb, torch, nx, nb, omega)
    D = cb.DDH(omega, ha, fem, nx, nx, 16)
    m = D.size()
    b = torch.empty(m, dtype=torch.float32, device="cuda")
    L = torch.zeros(m, dtype=torch.float32, device="cuda")
    D.rhs(f, b)
    tmp = torch.empty_like(b)
    D.action(b, tmp)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        D.action(b, tmp)
    e1.record()
    torch.cuda.synchronize()
    act_ms = e0.elapsed_time(e1) / 3
    res = {"nx": nx, "n_basis": nb, "omega": omega, "n_domains": D.info()["n_domains"], "nt": D.info()["nt"], "n_lambda": m,
           "action_ms": act_ms, "action_fp32_tflops": D.flops() / (act_ms * 1e-3) / 1e12}
    for name, mode in (("mgs", cb.MGS), ("cgs2", cb.CGS2)):
        L.zero_()
        t0 = time.perf_counter()
        out = cb.gmres(m, L, D, b, 20, 100, 1e-4, orth=mode)
        torch.cuda.synchronize()
        res["gmres_" + name] = {"seconds": time.perf_counter() - t0, "restarts": out.num_iter, "matvecs": out.num_matvec, "success": out.success}
    if drv:
        try:
            r = subprocess.run([drv, "time_ddh", str(nx), str(nb), repr(float(omega)), "3"], capture_output=True, text=True, timeout=900)
            res["reference_gpu_kernel"] = json.loads(r.stdout.strip().splitlines()[-1])
            res["action_speedup_vs_reference_kernel"] = res["reference_gpu_kernel"]["action_ms"] / act_ms
        except Exception as e:
            res["reference_gpu_kernel"] = "failed: %r" % (e,)
    return res


def helmholtz_example(cb, torch, drv, nx=128, nb=4, m=200, maxit=4, tol=1e-6):
    """examples/Helmholtz.cpp: uniform_rect(128), degree 3, omega = 2 pi 12.8, unpreconditioned FP64 GMRES(200); timed over the
    first maxit - 1 restart cycles (the full solve takes far longer), library gmres (both orthogonalisations) against the reference
    library's gmres + operators on the same GPU."""
    import tempfile
    from oracle.rdmp import read_rdmp
    omega = 2 * np.pi * nx / 10
    mesh = cb.Mesh2D.uniform_rect(nx, -1.0, 1.0, nx, -1.0, 1.0)
    fem = cb.H1Space(mesh, cb.Basis(nb))
    fs = cb.FaceSpace(fem, mesh.boundary_edges())
    n = fem.size()
    xy = fem.physical_coordinates()
    c = coef(xy[:, 0], xy[:, 1])
    dev = lambda a: torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device="cuda")
    A = cb.Helmholtz(omega, dev(c * c), dev(c[fs.global_indices()]), fem, fs)
    res = {"nx": nx, "n_basis": nb, "omega": omega, "n": 2 * n, "m": m, "restart_cycles": maxit - 1}
    ref = None
    if drv:
        with tempfile.NamedTemporaryFile(suffix=".bin") as fobj:
            subprocess.check_call([drv, "helm_gmres", "rect:%d" % nx, str(nb), repr(float(omega)), str(m), str(maxit), repr(tol), fobj.name], timeout=900)
            ref = read_rdmp(fobj.name)
        res["reference_library"] = {"seconds": float(ref["gmres_seconds"][0]), "restarts": int(ref["num_iter"][0]), "matvecs": int(ref["num_matvec"][0]),
                                    "rel_residual": float(ref["res_norm"][-1] / ref["res_norm"][0])}
    if ref is not None:
        b = dev(ref["b"])
    else:
        b = torch.zeros(2 * n, dtype=torch.float64, device="cuda")
        cb.LinearFunctional(fem).action(lambda X, Y: omega ** 2 / np.pi * torch.exp(-omega ** 2 * ((X + 0.5) ** 2 + Y ** 2)), b[:n])
    for name, mode in (("mgs", cb.MGS), ("cgs2", cb.CGS2)):
        U = torch.zeros(2 * n, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        o = cb.gmres(2 * n, U, A, b, m, maxit, tol, orth=mode)
        torch.cuda.synchronize()
        res["library_" + name] = {"seconds": time.perf_counter() - t0, "restarts": o.num_iter, "matvecs": o.num_matvec,
                                  "rel_residual": o.res_norm[-1] / o.res_norm[0], "reorth": o.reorth}
    return res


if __name__ == "__main__":
    main()
