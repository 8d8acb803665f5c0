"""Latency of ONE (or a few) LML+gradient evaluations -- the operating point of the Stan seam
(stan/gp_lml_stan.hpp -> gpb200_lml_grad, one theta per leapfrog step; models/fit_hyperparameters.stan:18-31
under pendulum_fit.R:206).  Device-resident inputs, CUDA events over `reps` back-to-back calls, results
With arguments "variants" the same measurement is repeated
under the tuning knobs (look-ahead off, panel widths, GEMM configurations) in child processes."""
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, ".")


def measure(sizes=((4096, 1), (2048, 1), (1024, 1), (100, 1), (4096, 4), (1024, 4), (100, 4)), reps=20):
    import torch
    from gp_b200 import capi
    dev = torch.device("cuda", 0)
    h = capi.Handle(0)
    stream = torch.cuda.current_stream(dev)
    h.set_stream(stream.cuda_stream)
    h.set_pointer_mode(True)
    out = {}
    for n, B in sizes:
        rng = np.random.default_rng(5)
        x = np.sort(rng.uniform(0, 0.05 * n, n))
        y = np.sin(x) + 0.5 * np.sin(3.1 * x) + 0.3 * rng.standard_normal(n)
        th = np.stack([np.abs(rng.standard_normal(B)) + 0.5, rng.gamma(4.0, 0.25, B) + 0.2, rng.uniform(0.1, 0.5, B)], axis=1)
        dx = torch.from_numpy(x).to(dev); dy = torch.from_numpy(y).to(dev); dth = torch.from_numpy(th).to(dev)
        lml = torch.empty(B, dtype=torch.float64, device=dev); grad = torch.empty(B, 3, dtype=torch.float64, device=dev)
        info = torch.zeros(B, dtype=torch.int32, device=dev)
        for _ in range(3):
            h.lml_grad_batched_device(n, B, dx, 0, dy, 0, dth, 0.0, True, lml, grad, info)
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            h.lml_grad_batched_device(n, B, dx, 0, dy, 0, dth, 0.0, True, lml, grad, info)
        e1.record(stream); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        rec = {"ms": round(ms, 4), "tflops": round(B * float(n) ** 3 / ms * 1e-9, 2), "info": int(info.abs().sum().item())}
        rec["lml0"] = float(lml[0].item())   # parity of this path is asserted in tests/ (the tools never touch the oracle)
        out["n=%d B=%d" % (n, B)] = rec
    h.close()
    return out


VARIANTS = [
    ("default", {}),
    ("no_lookahead", {"GPB200_LOOKAHEAD": "0"}),
    ("lookahead_pt2", {"GPB200_CHOL_PANEL": "2"}),
    ("lookahead_pt4", {"GPB200_CHOL_PANEL": "4"}),
    ("half8_only", {"GPB200_GEMM_CFG": "2"}),
    ("quarter_only", {"GPB200_GEMM_CFG": "3"}),
    ("no_graph", {"GPB200_NO_GRAPH": "1"}),
]

if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "child":
        print(json.dumps(measure()))
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "variants":
        res = {}
        for label, env in VARIANTS:
            e = dict(os.environ); e.update(env)
            r = subprocess.run([sys.executable, __file__, "child"], env=e, capture_output=True, text=True)
            res[label] = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else {"error": r.stderr[-1500:]}
            print(label, json.dumps(res[label]), flush=True)
        os.makedirs("gpurun_out", exist_ok=True)
        json.dump(res, open("gpurun_out/bench_latency_variants.json", "w"), indent=1)
    else:
        res = measure()
        print(json.dumps(res, indent=1))
        os.makedirs("gpurun_out", exist_ok=True)
        json.dump(res, open("gpurun_out/bench_latency.json", "w"), indent=1)
