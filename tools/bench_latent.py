"""The non-centred latent model (f = L z and its reverse sweep through the Cholesky) for B parameter states: the batched
calls against a loop of single-state calls.

  python tools/bench_latent.py [--reps 3] [--out profiles/bench_latent.json]

One forward + one backward per state, per call, timed with CUDA events after a warm-up of every shape; every repetition
draws new states, so no call finds the factor of its state cached.  Three ways:
  a) loop     gpb200_latent_forward / gpb200_latent_backward per state, host pointers (what a caller had before)
  b) batched  gpb200_latent_forward_batched / _backward_batched, host pointers
  c) device   the batched calls in device-pointer mode, fbar = (y - f) / sigma^2 computed by torch in between
Shapes: n = 100 on x = seq(0, 10, length = 100) with jitter 1e-10 (exact_gp.stan), n = 1438 on the Westbrook series with
jitter 1e-6 (westbrook_exact.stan), n = 4096 on the bench.py family (x = sort(U(0, 0.05 n))) with jitter 1e-6; B in
{1, 16, 64, 256}.  States: alpha ~ |N(0, 1)| + 0.5, rho ~ Gamma(4, 4) + 0.2 (seeded), z ~ N(0, 1), sigma = 0.3.
Reported per shape and B: ms per state (forward, backward, total), the rate on N^3/3 + N^3 flops per state, failed
states (info != 0), and the largest difference between a) and b) over the states that factor, relative to the largest
|entry| of a) for f and zbar and to |theta_bar| of a) per component.  The card name and power limit are read in the
same run and written beside the numbers."""
import argparse
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "tools"))

from bench_ard import card  # noqa: E402

SIGMA = 0.3


def shape(name):
    if name == "c1_n100":
        return np.linspace(0.0, 10.0, 100), 1e-10
    if name == "westbrook_n1438":
        w = np.load(os.path.join(HERE, "tests", "golden", "westbrook_xy.npz"))
        return np.sort(w["x"]), 1e-6
    rng = np.random.default_rng(5)
    return np.sort(rng.uniform(0.0, 0.05 * 4096, size=4096)), 1e-6


def states(n, B, seed):
    rng = np.random.default_rng(seed)
    th = np.stack([np.abs(rng.standard_normal(B)) + 0.5, rng.gamma(4.0, 0.25, B) + 0.2], axis=1)
    return th, rng.standard_normal((B, n))


class Timer:
    def __init__(self, torch):
        self.torch = torch
        self.ms = 0.0

    def __enter__(self):
        self.e0 = self.torch.cuda.Event(enable_timing=True)
        self.e1 = self.torch.cuda.Event(enable_timing=True)
        self.e0.record()
        return self

    def __exit__(self, *a):
        self.e1.record()
        self.e1.synchronize()
        self.ms += self.e0.elapsed_time(self.e1)


def run_loop(h, x, y, th, z, jitter, torch):
    from gp_b200 import capi
    B = th.shape[0]
    f = np.full_like(z, np.nan); zbar = np.full_like(z, np.nan); tb = np.full((B, 2), np.nan)
    tf, tbk = Timer(torch), Timer(torch)
    failed = 0
    for b in range(B):
        try:
            with tf:
                f[b] = h.latent_forward(x, th[b, 0], th[b, 1], jitter, z[b])
            with tbk:
                tb[b], zbar[b] = h.latent_backward(x, th[b, 0], th[b, 1], jitter, z[b], (y - f[b]) / SIGMA ** 2)
        except capi.NotPositiveDefiniteError:
            failed += 1
    return (f, tb, zbar), tf.ms, tbk.ms, failed


def run_batched(h, x, y, th, z, jitter, torch):
    tf, tbk = Timer(torch), Timer(torch)
    with tf:
        f, info = h.latent_forward_batched(x, th, jitter, z)
    with tbk:
        tb, zbar = h.latent_backward_batched((y - f) / SIGMA ** 2)
    return (f, tb, zbar), tf.ms, tbk.ms, int(np.count_nonzero(info))


class Device:
    def __init__(self, x, y, th, z, jitter, torch):
        from gp_b200 import capi
        dev = torch.device("cuda", 0)
        self.torch, self.jitter = torch, jitter
        self.B, self.n = z.shape
        self.x = torch.tensor(x, device=dev); self.y = torch.tensor(y, device=dev)
        self.th = torch.tensor(th, device=dev); self.z = torch.tensor(z, device=dev)
        self.f = torch.empty_like(self.z); self.zbar = torch.empty_like(self.z)
        self.tb = torch.empty((self.B, 2), dtype=torch.float64, device=dev)
        self.info = torch.empty(self.B, dtype=torch.int32, device=dev)
        self.h = capi.Handle(0)
        self.h.set_pointer_mode(True)
        self.h.set_stream(torch.cuda.current_stream().cuda_stream)

    def run(self):
        tf, tbk = Timer(self.torch), Timer(self.torch)
        with tf:
            self.h.latent_forward_batched_device(self.n, self.B, 1, self.x, 0, self.th, self.jitter, self.z, self.f, self.info)
        with tbk:
            fbar = (self.y - self.f) / SIGMA ** 2
            self.h.latent_backward_batched_device(self.n, self.B, 1, fbar, self.tb, self.zbar)
        return tf.ms, tbk.ms, int((self.info != 0).sum().item())

    def close(self):
        self.h.close()


def rel_diff(a, b, ok):
    if not ok.any():
        return None
    fa, fb = a[ok], b[ok]
    return float(np.max(np.abs(fa - fb)) / max(float(np.max(np.abs(fa))), 1e-300))


def bench(name, B, reps, torch):
    from gp_b200 import capi
    x, jitter = shape(name)
    n = x.shape[0]
    y = np.sin(x) + 0.5 * np.sin(3.1 * x)
    th, z = states(n, B, 1000 + B)   # the warm-up states; every repetition draws new ones (no call sees a state twice)
    flops = n ** 3 / 3.0 + float(n) ** 3
    out = {"n": n, "B": B, "jitter": jitter, "flops_per_state": flops}
    h = capi.Handle(0)
    dv = None
    try:
        run_loop(h, x, y, th[:1], z[:1], jitter, torch)
        run_batched(h, x, y, th, z, jitter, torch)
        dv = Device(x, y, th, z, jitter, torch)
        dv.run()
        torch.cuda.synchronize()
        res = {"loop": [0.0, 0.0], "batched": [0.0, 0.0], "device": [0.0, 0.0]}
        # the three ways alternate, on new states each time (the single-state calls cache the factor of their last state)
        for rep in range(reps):
            th, z = states(n, B, 2000 + 97 * rep + B)
            ra, fa, ba, fail_a = run_loop(h, x, y, th, z, jitter, torch)
            rb, fb, bb, fail_b = run_batched(h, x, y, th, z, jitter, torch)
            dv.th.copy_(torch.from_numpy(th)); dv.z.copy_(torch.from_numpy(z))
            fc, bc, fail_c = dv.run()
            for k, (tf, tbk) in (("loop", (fa, ba)), ("batched", (fb, bb)), ("device", (fc, bc))):
                res[k][0] += tf; res[k][1] += tbk
        for k, (tf, tbk) in res.items():
            fwd, bwd = tf / reps / B, tbk / reps / B
            out[k] = {"ms_per_state_forward": fwd, "ms_per_state_backward": bwd, "ms_per_state": fwd + bwd,
                      "gflops": flops / ((fwd + bwd) * 1e-3) / 1e9}
        out["failed"] = {"loop": fail_a, "batched": fail_b, "device": fail_c}
        ok = np.all(np.isfinite(ra[1]), axis=1) & np.all(np.isfinite(rb[1]), axis=1)
        tdiff = None
        if ok.any():
            tdiff = float(np.max(np.abs(ra[1][ok] - rb[1][ok]) / np.maximum(np.abs(ra[1][ok]), 1e-300)))
        out["max_rel_diff_loop_vs_batched"] = {"f": rel_diff(ra[0], rb[0], ok), "zbar": rel_diff(ra[2], rb[2], ok),
                                               "theta_bar": tdiff}
        out["speedup_batched_over_loop"] = out["loop"]["ms_per_state"] / out["batched"]["ms_per_state"]
        out["speedup_device_over_loop"] = out["loop"]["ms_per_state"] / out["device"]["ms_per_state"]
    except capi.GpB200Error as e:
        out["not_run"] = str(e)
    finally:
        if dv is not None:
            dv.close()
        h.close()
        torch.cuda.empty_cache()
    return out


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--shapes", default="c1_n100,westbrook_n1438,bench_n4096")
    ap.add_argument("--batches", default="1,16,64,256")
    ap.add_argument("--out", default=os.path.join(HERE, "profiles", "bench_latent.json"))
    a = ap.parse_args()
    res = {"card": card(), "reps": a.reps, "runs": []}
    for name in a.shapes.split(","):
        for B in (int(v) for v in a.batches.split(",")):
            r = bench(name, B, a.reps, torch)
            r["shape"] = name
            res["runs"].append(r)
            print(name, B, json.dumps({k: r.get(k) for k in ("failed", "speedup_batched_over_loop", "speedup_device_over_loop",
                                                             "max_rel_diff_loop_vs_batched", "not_run")}), flush=True)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"], "out": a.out}))


if __name__ == "__main__":
    main()
