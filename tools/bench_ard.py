"""ARD LML + gradient (gpb200_lml_grad_ard_batched) against the SE route at D = 1, in one process.

  python tools/bench_ard.py [--reps 5] [--out profiles/bench_ard.json]

Device-pointer mode, CUDA events on torch's current stream, every shape warmed up first.  It times
  - N = 4096, B = 256 for D in 1, 2, 4, 8 (one call = B LML + gradient evaluations), and the per-class kernel times of
    gpb200_set_profiling for one call of each (GEMM, Gram, other = everything else), in a separate pass;
  - B = 1 latency at N = 1024 and 4096 for D = 1 and D = 8;
  - the comparison: gpb200_lml_grad_batched at D = 1 on the same inputs, on a GPB200_ENVELOPE=0 handle (the dense route
    the ARD kind also takes) and on the default handle (tile envelope + selected inverse).
One B = 256, N = 4096 call works on ~64 GB of factors: far beyond the 126 MB L2.  The card name and power
limit are read in the same run and written beside the numbers."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, HERE)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as e:  # the numbers stay valid; say the card could not be read
        return {"error": repr(e)}


def make_handle(env=None):
    from gp_b200 import capi
    env = env or {}
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return capi.Handle(0)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def inputs(n, D, B, seed=3):
    import torch
    rng = np.random.default_rng(seed)
    X = rng.uniform(0.0, 0.05 * n, size=(D, n))          # column-major n x D, shared by the batch
    y = np.sin(X.sum(axis=0)) + 0.3 * rng.standard_normal(n)
    th = np.empty((B, D + 2))
    th[:, 0] = np.abs(rng.standard_normal(B)) + 0.1
    th[:, 1:D + 1] = rng.gamma(4.0, 0.25, size=(B, D)) * np.sqrt(D)
    th[:, D + 1] = rng.uniform(0.1, 0.5, size=B)
    dev = torch.device("cuda", 0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    return {"X": t(X), "y": t(y), "th": t(th), "lml": torch.empty(B, dtype=torch.float64, device=dev),
            "grad": torch.empty(B * (D + 2), dtype=torch.float64, device=dev),
            "info": torch.zeros(B, dtype=torch.int32, device=dev)}


def call(h, kind, n, D, B, a):
    if kind == "ard":
        h.lml_grad_ard_batched_device(n, D, B, a["X"], 0, a["y"], 0, a["th"], 0.0, True, a["lml"], a["grad"], a["info"])
    else:
        h.lml_grad_batched_device(n, B, a["X"], 0, a["y"], 0, a["th"], 0.0, True, a["lml"], a["grad"], a["info"])


def timed(h, kind, n, D, B, a, reps):
    import torch
    call(h, kind, n, D, B, a)  # warm-up: modules, task lists, graphs, workspace
    call(h, kind, n, D, B, a)
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        call(h, kind, n, D, B, a)
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    assert int(a["info"].max().item()) == 0 and int(a["info"].min().item()) == 0
    return {"ms_median": float(np.median(ms)), "ms_min": float(np.min(ms)), "ms_max": float(np.max(ms)), "reps": reps}


def classes(h, kind, n, D, B, a):
    import torch
    h.set_profiling(True)
    call(h, kind, n, D, B, a)
    torch.cuda.synchronize()
    prof = h.get_profile()
    h.set_profiling(False)
    gemm, gram = prof["gemm"][0], prof["gram"][0]
    other = sum(v[0] for k, v in prof.items() if k not in ("gemm", "gram"))
    return {"gemm_ms": gemm, "gram_ms": gram, "other_ms": other}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(HERE, "profiles", "bench_ard.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_ard: no GPU (nothing is measured on the CPU)")
    stream = torch.cuda.current_stream().cuda_stream
    handles = {"default": make_handle(), "dense_se": make_handle({"GPB200_ENVELOPE": "0"})}
    for h in handles.values():
        h.set_stream(stream)
        h.set_pointer_mode(True)
    res = {"card": card(), "what": "ms per call (CUDA events, device pointers, shared X and y); evals/s = B / s",
           "batched": {}, "latency": {}}
    n, B = 4096, 256
    for D in (1, 2, 4, 8):
        a = inputs(n, D, B)
        r = timed(handles["default"], "ard", n, D, B, a, args.reps)
        r["evals_per_s"] = B / (r["ms_median"] * 1e-3)
        r.update(classes(handles["default"], "ard", n, D, B, a))
        res["batched"]["ard_D%d" % D] = r
        if D == 1:
            for name in ("dense_se", "default"):
                rs = timed(handles[name], "se", n, 1, B, a, args.reps)
                rs["evals_per_s"] = B / (rs["ms_median"] * 1e-3)
                rs.update(classes(handles[name], "se", n, 1, B, a))
                res["batched"]["se_%s" % name] = rs
        del a
        torch.cuda.empty_cache()
        print(json.dumps({k: res["batched"][k] for k in res["batched"] if k.endswith("D%d" % D)}), flush=True)
    for n1 in (1024, 4096):
        for D in (1, 8):
            a = inputs(n1, D, 1)
            res["latency"]["ard_D%d_N%d" % (D, n1)] = timed(handles["default"], "ard", n1, D, 1, a, 4 * args.reps)
            if D == 1:
                for name in ("dense_se", "default"):
                    res["latency"]["se_%s_N%d" % (name, n1)] = timed(handles[name], "se", n1, 1, 1, a, 4 * args.reps)
    b = res["batched"]
    res["ard_D1_over_dense_se"] = b["ard_D1"]["ms_median"] / b["se_dense_se"]["ms_median"]
    res["ard_D8_minus_D1_ms"] = {"total": b["ard_D8"]["ms_median"] - b["ard_D1"]["ms_median"],
                                 "gram": b["ard_D8"]["gram_ms"] - b["ard_D1"]["gram_ms"],
                                 "gemm": b["ard_D8"]["gemm_ms"] - b["ard_D1"]["gemm_ms"]}
    for h in handles.values():
        h.set_pointer_mode(False)
        h.close()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
