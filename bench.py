#!/usr/bin/env python
"""bench.py -- headline benchmark of the GP hot path on B200.

Metric (BASELINE.json): LML + gradient evaluations per second at N = 4096.
A "step" is one pass of the fused path (Gram -> Cholesky -> inverse -> LML + gradient) over one
batch of B = 256 independent hyper-parameter draws per GPU on synthetic inputs (SURVEY 8d
"Headline"); draws are sharded over GPUs with no data-path collective (weak scaling).

  value     evaluations/s with inputs resident in HBM, timed with CUDA events on the launching
            stream, max over ranks
  e2e       the same metric through the C ABI with HOST buffers (pinned), H2D/D2H inside the timer
  roofline  the dominant kernel (DMMA tile GEMM): algorithmic FP64 flops / event-timed duration vs
            the measured DMMA peak (profiles/fp64_peak_r01.json; MEASURED_PEAKS.json has no FP64)
  cpu_baseline  the CPU oracle (LAPACK route, all host cores) on a bounded sample, rank 0, N=1 only

`--impl reference` times the reference's CPU path instead: the reference itself (R + Stan Math +
Eigen) cannot be built or run in this image, so this is the oracle port (kind "port").

`--dump-outputs DIR` writes what the last timed step returned to DIR/lml.npy (draws,), DIR/grad.npy
(draws, 3) and DIR/info.npy (draws,), all float64, draws of every rank in rank order.  The inputs are
seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N = 4096
DRAWS_PER_GPU = 256
METRIC = "lml_grad_evals_per_sec_n4096"
UNIT = "evals/s"
TILE = 128


def fp64_peak():
    """Measured FP64 tensor (DMMA) peak of this pool's B200 in TFLOP/s, and where it came from."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            mp = json.load(f)
        if "fp64_tflops" in mp:
            return float(mp["fp64_tflops"]), "MEASURED_PEAKS.json fp64_tflops"
    except Exception:
        pass
    try:
        with open(os.path.join(ROOT, "profiles", "fp64_peak_r01.json")) as f:
            return float(json.load(f)["fp64_dmma_tflops"]), "profiles/fp64_peak_r01.json (DMMA issue-rate microbenchmark, round 1)"
    except Exception:
        return 37.0, "fallback 37.0 (148 SM x 1.965 GHz x 128 flop/clk)"


def gemm_algorithmic_flops(n):
    """Algorithmic flops of one LML+grad evaluation that are carried by the DMMA GEMM launches:
    N^3 (SURVEY 8d: N^3/3 POTRF + 2N^3/3 inverse) minus what the 128-wide panel kernels do
    (POTRF tiles nt*T^3/3, TRSM tiles nt(nt-1)/2*T^3, tile inverses nt*T^3/3)."""
    nt = (n + TILE - 1) // TILE
    t3 = float(TILE) ** 3
    return float(n) ** 3 - t3 * (nt / 3.0 + nt * (nt - 1) / 2.0 + nt / 3.0)


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""
    BAD = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown"}
    NOTE = {0x4: "sw_power_cap", 0x80: "hw_power_brake", 0x2: "applications_clocks_setting"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = threading.Event()
        self.sm = []
        self.reasons = set()
        self.sm_max = None
        self.ok = False

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.index
            if vis:
                try:
                    idx = int(vis.split(",")[self.index])
                except Exception:
                    pass
            dev = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(dev, pynvml.NVML_CLOCK_SM)
            self.ok = True
            while not self.stop_flag.is_set():
                self.sm.append(pynvml.nvmlDeviceGetClockInfo(dev, pynvml.NVML_CLOCK_SM))
                try:
                    r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(dev)
                except Exception:
                    r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(dev)
                for bit, name in list(self.BAD.items()) + list(self.NOTE.items()):
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.1)
        except Exception as e:  # pragma: no cover
            self.error = repr(e)

    def result(self):
        self.stop_flag.set()
        self.join(timeout=2.0)
        if not self.ok or not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["nvml_unavailable"]}
        s = sorted(self.sm)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons)}


def synth_inputs(rank):
    """Synthetic workload of SURVEY 8d: x = sort(U(0, 0.05 N)), y = sin(x) + 0.5 sin(3.1 x) + 0.3 eps;
    theta draws alpha ~ |N(0,1)| + 0.1, rho ~ Gamma(4,4) (fit_hyperparameters.stan:27), sigma ~ U(.1,.5)."""
    import numpy as np
    rng = np.random.default_rng(5)
    x = np.sort(rng.uniform(0.0, 0.05 * N, size=N))
    y = np.sin(x) + 0.5 * np.sin(3.1 * x) + 0.3 * rng.standard_normal(N)
    r2 = np.random.default_rng(1000 + rank)
    theta = np.stack([np.abs(r2.standard_normal(DRAWS_PER_GPU)) + 0.1, r2.gamma(4.0, 0.25, DRAWS_PER_GPU),
                      r2.uniform(0.1, 0.5, DRAWS_PER_GPU)], axis=1)
    return x, y, theta


def synth_small(n, B, seed=5):
    """The same synthetic family at another size (latency extras)."""
    import numpy as np
    rng = np.random.default_rng(seed)
    x = np.sort(rng.uniform(0.0, 0.05 * n, size=n))
    y = np.sin(x) + 0.5 * np.sin(3.1 * x) + 0.3 * rng.standard_normal(n)
    theta = np.stack([np.abs(rng.standard_normal(B)) + 0.5, rng.gamma(4.0, 0.25, B) + 0.2, rng.uniform(0.1, 0.5, B)], axis=1)
    return x, y, theta


def measure_latency(h, dev, stream, reps=20):
    """Latency of ONE evaluation (B = 1) and of a handful (B = 4): the operating point of the Stan seam, where NUTS
    asks for one log_prob_grad per leapfrog step per chain (models/fit_hyperparameters.stan:18-31 under
    pendulum_fit.R:206).  Device-resident inputs, CUDA events over `reps` back-to-back calls after 3 warm-ups."""
    import torch
    out = {}
    for n in (4096, 1024, 100):
        for B in (1, 4):
            x, y, th = synth_small(n, B)
            dx = torch.from_numpy(x).to(dev); dy = torch.from_numpy(y).to(dev); dth = torch.from_numpy(th).to(dev)
            lml = torch.empty(B, dtype=torch.float64, device=dev); grad = torch.empty(B, 3, dtype=torch.float64, device=dev)
            info = torch.zeros(B, dtype=torch.int32, device=dev)
            for _ in range(3):
                h.lml_grad_batched_device(n, B, dx, 0, dy, 0, dth, 0.0, True, lml, grad, info)
            torch.cuda.synchronize(dev)
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(reps):
                h.lml_grad_batched_device(n, B, dx, 0, dy, 0, dth, 0.0, True, lml, grad, info)
            e1.record(stream)
            torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1) / reps
            out["n%d_b%d" % (n, B)] = {"ms_per_call": round(ms, 4), "tflops": round(B * float(n) ** 3 / ms * 1e-9, 2),
                                       "all_pd": int(info.abs().sum().item()) == 0,
                                       "_check": (x, y, th, lml.cpu().numpy().copy(), grad.cpu().numpy().copy())}
    return out


def measure_block_cyclic(h, dev, world, rank, sizes=(32768, 16384, 8192)):
    """Config 5 (SURVEY 8e): ONE large exact GP, LML + gradient (models/fit_hyperparameters.stan:19-31 semantics), factor
    block-column-cyclic over the ranks with the panel broadcasts enqueued from C (gpb200_mg_bcast -> ncclBroadcast), exact
    distributed gradient.  Time = factorisation + gradient, CUDA events, max over ranks, best of 2 after a warm-up."""
    import importlib.util
    import numpy as np
    import torch
    spec = importlib.util.spec_from_file_location("bench_block_cyclic", os.path.join(ROOT, "tools", "bench_block_cyclic.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    from gp_b200.block_cyclic import GpuPanelBackend
    be = GpuPanelBackend(h, dev).init_comm()
    out = {}
    try:
        for n in sizes:
            pc = 256 if n // world <= 2048 else 512   # narrower panels when each rank holds few of them (measured: 8 ranks, N = 16 384)
            rec, (x, y, theta) = mod.run_one(n, pc, be, h, dev, world, rank, reps=2)
            rec.pop("grad", None)
            if rank == 0 and n <= 8192:   # checker leg: the oracle at a size it finishes in seconds
                from oracle import gp_oracle as _o
                from threadpoolctl import threadpool_limits
                with threadpool_limits(limits=os.cpu_count() or 1):
                    rv, rg = _o.lml_grad_lapack(x, y, *theta)
                rec["relerr_lml_vs_oracle"] = float(abs(rec["lml"] - rv) / abs(rv))
                rec["relerr_grad_vs_oracle"] = float(np.max(np.abs(np.asarray(rec["grad_full"]) - rg)) / np.max(np.abs(rg)))
            rec.pop("grad_full", None)
            out["n%d" % n] = rec
    finally:
        be.close_comm()
        h.set_stream(torch.cuda.current_stream(dev).cuda_stream)
    return out


def cpu_reference_evals_per_sec(n_evals, threads):
    """Times the CPU oracle (LAPACK route) on `n_evals` draws of the N=4096 workload with `threads`
    BLAS threads (torchrun exports OMP_NUM_THREADS=1, so the pool size is set explicitly)."""
    from oracle import gp_oracle as o
    from threadpoolctl import threadpool_limits
    x, y, theta = synth_inputs(0)
    out = []
    with threadpool_limits(limits=threads):
        t0 = time.perf_counter()
        for b in range(n_evals):
            out.append(o.lml_grad_lapack(x, y, *theta[b]))
        dt = time.perf_counter() - t0
    return n_evals / dt, dt, out


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, outputs, world, rank):
    """Writes the device tensors `outputs` (name -> tensor with the draws on axis 0) as float64 .npy files under
    `path`, each gathered over the ranks in rank order; rank 0 writes."""
    import numpy as np
    import torch
    import torch.distributed as dist
    host = {}
    for name, t in outputs.items():
        if world > 1:
            parts = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(parts, t.contiguous())
            t = torch.cat(parts)
        host[name] = t.cpu().numpy().astype(np.float64)
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d-byte limit; use fewer --draws" % (total, DUMP_LIMIT_BYTES))
    if rank == 0:
        os.makedirs(path, exist_ok=True)
        for name, a in host.items():
            np.save(os.path.join(path, name + ".npy"), a)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    # all host threads: torchrun pins OMP_NUM_THREADS=1 for its children, undo that before NumPy loads
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = str(threads)
    per_step = 2
    for _ in range(args.warmup):
        cpu_reference_evals_per_sec(1, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_reference_evals_per_sec(per_step, threads)
    dt = time.perf_counter() - t0
    v = args.steps * per_step / dt
    sample = "%d LML+grad evaluations per step at N=%d (oracle.lml_grad_lapack: OpenBLAS dpotrf+dpotri, %d threads)" % (
        per_step, N, threads)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "lml+grad, 1-D SE kernel, N=4096, independent theta draws (CPU sample of %d draws/step)" % per_step,
                       "n": N, "draws_per_step": per_step},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "the reference (R + Stan Math + Eigen) cannot be built here; this is the CPU oracle port"}
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="gpb200", choices=["gpb200", "reference"])
    ap.add_argument("--draws", type=int, default=DRAWS_PER_GPU)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write lml, grad and info of the last timed step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from gp_b200 import capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback for the product path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.draws
    W = max(args.warmup, 3)
    K = args.steps

    h = capi.Handle(local_rank)
    stream = torch.cuda.current_stream(dev)
    h.set_stream(stream.cuda_stream)

    x, y, theta = synth_inputs(rank)
    dx = torch.from_numpy(x).to(dev)
    dy = torch.from_numpy(y).to(dev)
    dth = torch.from_numpy(theta).to(dev)
    dlml = torch.empty(B, dtype=torch.float64, device=dev)
    dgrad = torch.empty(B, 3, dtype=torch.float64, device=dev)
    dinfo = torch.zeros(B, dtype=torch.int32, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---------------- value: HBM-resident inputs, device-pointer mode --------------------------
    h.set_pointer_mode(True)

    def step_device():
        h.lml_grad_batched_device(N, B, dx, 0, dy, 0, dth, 0.0, True, dlml, dgrad, dinfo)

    for _ in range(W):
        step_device()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    h.set_profiling(True)
    h.lib.gpb200_set_flop_counting(h._h, 1)
    launches0 = h.launch_count()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(K):
        step_device()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = h.launch_count() - launches0
    prof = h.get_profile()
    h.set_profiling(False)
    executed_flops = float(h.lib.gpb200_executed_gemm_flops(h._h))
    h.lib.gpb200_set_flop_counting(h._h, 0)
    clocks = sampler.result()
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * B * K / (ms_max * 1e-3)
    assert int(dinfo.abs().sum().item()) == 0, "a synthetic draw was not positive definite"
    lml_dev = dlml.cpu().numpy().copy()
    if args.dump_outputs:   # before the LML-only pass below overwrites dlml
        dump_outputs(args.dump_outputs, {"lml": dlml, "grad": dgrad, "info": dinfo}, world, rank)

    # ---------------- second half of BASELINE's metric: Cholesky FP64 TFLOP/s vs peak ------------
    # the LML-only pass (Gram -> tiled Cholesky -> forward substitution -> log-det/quadratic form) of
    # the same batch, N^3/3 flops per evaluation (LAPACK convention), timed apart from the headline
    def step_chol():
        h.lml_grad_batched_device(N, B, dx, 0, dy, 0, dth, 0.0, False, dlml, dgrad, dinfo)

    step_chol()
    barrier()
    c0 = torch.cuda.Event(enable_timing=True)
    c1 = torch.cuda.Event(enable_timing=True)
    kc = max(1, min(K, 3))
    c0.record(stream)
    for _ in range(kc):
        step_chol()
    c1.record(stream)
    barrier()
    t = torch.tensor([c0.elapsed_time(c1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    chol_ms = float(t.item()) / kc
    chol_tflops = B * float(N) ** 3 / 3.0 / (chol_ms * 1e-3) * 1e-12   # per GPU

    # ---------------- e2e: host (pinned) buffers through the C ABI ----------------------------
    h.set_pointer_mode(False)
    hx = torch.from_numpy(x).pin_memory()
    hy = torch.from_numpy(y).pin_memory()
    hth = torch.from_numpy(theta).pin_memory()
    hlml = torch.empty(B, dtype=torch.float64).pin_memory()
    hgrad = torch.empty(B, 3, dtype=torch.float64).pin_memory()
    hinfo = torch.zeros(B, dtype=torch.int32).pin_memory()

    def step_host():
        rc = h.lib.gpb200_lml_grad_batched(h._h, N, B, hx.data_ptr(), 0, hy.data_ptr(), 0, hth.data_ptr(), 0.0, 1,
                                           hlml.data_ptr(), hgrad.data_ptr(), hinfo.data_ptr())
        if rc != 0:
            raise RuntimeError("lml_grad_batched failed: %d" % rc)

    step_host()
    barrier()
    e2 = torch.cuda.Event(enable_timing=True)
    e3 = torch.cuda.Event(enable_timing=True)
    e2.record(stream)
    t0 = time.perf_counter()
    for _ in range(K):
        step_host()
    e3.record(stream)
    torch.cuda.synchronize(dev)
    wall_ms = (time.perf_counter() - t0) * 1e3
    e2e_ms = max(e2.elapsed_time(e3), wall_ms)
    t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * K / (float(t.item()) * 1e-3)
    h2d = (x.nbytes + y.nbytes + theta.nbytes)
    d2h = B * 8 + B * 24 + B * 4
    assert np.allclose(hlml.numpy(), lml_dev, rtol=1e-12, atol=0)

    # ---------------- latency extras: one evaluation and a handful (rank 0; the others wait) -----------
    h.set_pointer_mode(True)
    latency = measure_latency(h, dev, stream) if rank == 0 else None
    h.set_pointer_mode(False)
    barrier()

    # ---------------- checker leg (untimed): every rank compares its FIRST and LAST draw of the timed step, as the
    # host saw them through the C ABI, with the CPU oracle (the only use of oracle/ in this arm besides cpu_baseline)
    from oracle import gp_oracle as _o
    from threadpoolctl import threadpool_limits
    worst = np.zeros(2)
    with threadpool_limits(limits=max(1, (os.cpu_count() or 1) // world)):
        for b in sorted({0, B - 1}):
            rv, rg = _o.lml_grad_lapack(x, y, *theta[b])
            worst[0] = max(worst[0], abs(hlml.numpy()[b] - rv) / abs(rv))
            worst[1] = max(worst[1], float(np.max(np.abs(hgrad.numpy()[b] - rg)) / np.max(np.abs(rg))))
    wt = torch.from_numpy(worst).to(dev)
    if world > 1:
        dist.all_reduce(wt, op=dist.ReduceOp.MAX)
    worst = wt.cpu().numpy()
    assert worst[0] <= 1e-9 and worst[1] <= 1e-9, "rank-level parity check against the oracle failed: %r" % (worst,)
    parity = {"what": "first and last draw of every rank's timed batch vs oracle.lml_grad_lapack, relative error, max over ranks",
              "ranks": world, "draws_checked_per_rank": len({0, B - 1}), "max_relerr_lml": float(worst[0]),
              "max_relerr_grad": float(worst[1]), "tolerance": 1e-9}

    # ---------------- roofline of the dominant kernel -------------------------------------------
    peak, peak_src = fp64_peak()
    gemm_ms, gemm_count = prof["gemm"]
    gemm_flops_step = gemm_algorithmic_flops(N) * B
    achieved = gemm_flops_step * K / (gemm_ms * 1e-3) * 1e-12 if gemm_ms > 0 else None
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            traffic = json.load(f).get("gemm_dram_bytes_per_launch")
    except Exception:
        pass
    roofline = {"bound": "tensor", "kernel": "gpb::gemm_tile_kernel (DMMA.8x8x4 FP64 tile GEMM, all launches of the step)",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": (achieved / peak) if achieved else None,
                "traffic": traffic, "peak_source": peak_src + " -- of measured",
                "launches_per_step": gemm_count // max(K, 1), "kernel_ms_per_step": gemm_ms / K,
                "executed_over_algorithmic": executed_flops / (gemm_flops_step * K) if gemm_flops_step else None,
                "executed_tflops": executed_flops / (gemm_ms * 1e-3) * 1e-12 if gemm_ms > 0 else None,
                "kernel_share_of_step": gemm_ms / ms if ms > 0 else None,
                "whole_step_tflops": value / world * float(N) ** 3 * 1e-12,
                "whole_step_frac": value / world * float(N) ** 3 * 1e-12 / peak,
                "other_kernels_ms_per_step": {k: v[0] / K for k, v in prof.items() if k != "gemm"}}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "lml+grad (Gram->Cholesky->inverse->fused trace), 1-D SE kernel, N=4096, %d independent "
                                   "theta draws per GPU per step (SURVEY 8d headline)" % B,
                       "n": N, "draws_per_gpu": B, "parallelism": "draws sharded over %d GPU(s), no collective" % world,
                       "l2": "working set %.1f GB per step >> 126 MB L2 (no flush needed)" % (B * 2 * N * N * 8 / 1e9)},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches), "roofline": roofline}
    peak_c, _ = fp64_peak()
    line["cholesky"] = {"tflops_per_gpu": chol_tflops, "peak": peak_c, "frac": chol_tflops / peak_c, "ms_per_step": chol_ms,
                        "what": "LML-only pass of the same batch (Gram + left-looking tiled Cholesky + forward "
                                "substitution), N^3/3 flops per evaluation, CUDA events, max over ranks"}

    line["parity"] = parity
    if world > 1:
        bc = measure_block_cyclic(h, dev, world, rank)
        if rank == 0:
            line["block_cyclic"] = dict(bc, what="config 5: one exact GP of size N, LML+gradient, block-column-cyclic Cholesky with "
                                                 "NCCL panel broadcasts enqueued from C + exact distributed gradient; frac = N^3 / time / "
                                                 "(n_gpus x measured FP64 peak)")
    if latency is not None:
        if world == 1 and not args.no_cpu_baseline:   # the small latency cases are checked against the oracle too
            for k, rec in latency.items():
                lx, ly, lth, llml, lgrad = rec["_check"]
                if lx.shape[0] <= 1024:
                    rv, rg = _o.lml_grad(lx, ly, *lth[0])
                    assert abs(llml[0] - rv) <= 1e-9 * abs(rv) and np.max(np.abs(lgrad[0] - rg)) <= 1e-9 * np.max(np.abs(rg)), k
        for rec in latency.values():
            rec.pop("_check")
        line["latency"] = dict(latency, what="device-resident LML+gradient latency per call, B = 1 and B = 4 (CUDA-graph replay, "
                                             "look-ahead Cholesky with fused POTRF+TRSM launches, quarter- and fine-tile GEMM CTAs), CUDA events, rank 0")
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        n_evals = 8
        v, dt, out = cpu_reference_evals_per_sec(n_evals, threads)
        # the timed GPU results must equal the oracle's on the same draws (1e-9 relative)
        for b in range(n_evals):
            assert abs(out[b][0] - lml_dev[b]) <= 1e-9 * abs(out[b][0]), (b, out[b][0], lml_dev[b])
            g = hgrad.numpy()[b]
            assert np.max(np.abs(g - out[b][1])) <= 1e-9 * np.max(np.abs(out[b][1])), (b, g, out[b][1])
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": "%d of the %d draws of one step at N=%d, oracle.lml_grad_lapack (OpenBLAS "
                                          "dpotrf+dpotri, %d threads), %.1f s; GPU results checked against them to 1e-9" % (
                                              n_evals, B, N, threads, dt)}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    h.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
