"""Per-group GPs of different sizes: gpb200_lml_grad_ragged against the two ways a caller does it without it.

  python tools/bench_ragged.py [--reps 5] [--out profiles/bench_ragged.json]

Device-pointer mode, CUDA events on torch's current stream, every call warmed up first.  Each group is drawn from the
bench.py synthetic family at its own size (x = sort(U(0, 0.05 n)), y = sin(x) + 0.5 sin(3.1 x) + 0.3 eps, theta with
alpha ~ |N(0,1)| + 0.5, rho ~ Gamma(4,4) + 0.2, sigma ~ U(.1,.5)), seeded per group.  Workloads:
  a) 256 groups, sizes log-uniform in [32, 2048]                     (the per-player model with realistic sizes)
  b) 32 groups of 1024, also timed with one gpb200_lml_grad_batched   (what the ragged machinery costs)
  c) the Westbrook series (N = 1438, sorted, jitter 1e-6) + 63 groups of 64..512
For each: ms per call, evals/s, sum n_b^3 / s, kernel launches per call, and the alternatives
  loop      one gpb200_lml_grad_batched call per group (B = 1)
  per_size  one gpb200_lml_grad_batched call per distinct size (groups of equal size batched together).
The card name and power limit are read in the same run and written beside the numbers."""
import argparse
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "tools"))

from bench_ard import card  # noqa: E402


def family(n, seed):
    rng = np.random.default_rng(seed)
    x = np.sort(rng.uniform(0.0, 0.05 * n, size=n))
    y = np.sin(x) + 0.5 * np.sin(3.1 * x) + 0.3 * rng.standard_normal(n)
    th = [abs(rng.standard_normal()) + 0.5, rng.gamma(4.0, 0.25) + 0.2, rng.uniform(0.1, 0.5)]
    return x, y, th


def workload(name):
    if name == "a":
        sizes = np.round(np.exp(np.random.default_rng(7).uniform(np.log(32), np.log(2048), 256))).astype(int)
        groups = [family(int(n), 100 + g) for g, n in enumerate(sizes)]
        return groups, 0.0
    if name == "b":
        return [family(1024, 200 + g) for g in range(32)], 0.0
    w = np.load(os.path.join(HERE, "tests", "golden", "westbrook_xy.npz"))
    order = np.argsort(w["x"], kind="stable")
    groups = [(w["x"][order], (w["y"] - w["y"].mean())[order], [0.5, 0.2, 0.45])]
    sizes = np.random.default_rng(9).integers(64, 513, 63)
    groups += [family(int(n), 300 + g) for g, n in enumerate(sizes)]
    return groups, 1e-6


class Ragged:
    def __init__(self, groups, jitter):
        import torch
        dev = torch.device("cuda", 0)
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)  # noqa: E731
        self.B = len(groups)
        self.jitter = jitter
        self.offsets = np.concatenate([[0], np.cumsum([len(g[0]) for g in groups])]).astype(np.int64)
        self.x = t(np.concatenate([g[0] for g in groups]))
        self.y = t(np.concatenate([g[1] for g in groups]))
        self.th = t(np.array([g[2] for g in groups]))
        self.lml = torch.empty(self.B, dtype=torch.float64, device=dev)
        self.grad = torch.empty(3 * self.B, dtype=torch.float64, device=dev)
        self.info = torch.zeros(self.B, dtype=torch.int32, device=dev)
        # the uniform calls' view of the same inputs: per distinct size, the groups stacked row by row
        self.by_size = {}
        for b, g in enumerate(groups):
            self.by_size.setdefault(len(g[0]), []).append(b)
        self.stacks = {}
        for n, idx in self.by_size.items():
            self.stacks[n] = (t(np.stack([groups[b][0] for b in idx])), t(np.stack([groups[b][1] for b in idx])),
                              t(np.array([groups[b][2] for b in idx])), torch.empty(len(idx), dtype=torch.float64, device=dev),
                              torch.empty(3 * len(idx), dtype=torch.float64, device=dev),
                              torch.zeros(len(idx), dtype=torch.int32, device=dev))
        self.singles = [(t(g[0]), t(g[1]), t(np.array([g[2]]))) for g in groups]
        self.work = float(sum(float(len(g[0])) ** 3 for g in groups))

    def ragged(self, h):
        h.lml_grad_ragged_device(self.B, self.offsets, self.x, self.y, self.th, self.jitter, True, self.lml, self.grad,
                                 self.info)

    def per_size(self, h):
        for n, (x, y, th, lml, grad, info) in self.stacks.items():
            h.lml_grad_batched_device(n, len(self.by_size[n]), x, n, y, n, th, self.jitter, True, lml, grad, info)

    def loop(self, h):
        for b, (x, y, th) in enumerate(self.singles):
            h.lml_grad_batched_device(x.numel(), 1, x, 0, y, 0, th, self.jitter, True, self.lml[b:b + 1],
                                      self.grad[3 * b:3 * b + 3], self.info[b:b + 1])


def timed(h, fn, reps, B, work):
    import torch
    fn(h)
    fn(h)
    torch.cuda.synchronize()
    l0 = h.launch_count()
    fn(h)
    torch.cuda.synchronize()
    launches = h.launch_count() - l0
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn(h)
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    med = float(np.median(ms))
    return {"ms_median": med, "ms_min": float(np.min(ms)), "ms_max": float(np.max(ms)), "reps": reps,
            "evals_per_s": B / (med * 1e-3), "sum_n3_per_s": work / (med * 1e-3), "launches_per_call": int(launches)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(HERE, "profiles", "bench_ragged.json"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_ragged: no GPU (nothing is measured on the CPU)")
    from gp_b200 import capi
    h = capi.Handle(0)
    h.set_stream(torch.cuda.current_stream().cuda_stream)
    h.set_pointer_mode(True)
    res = {"card": card(), "what": "ms per call of all B groups (CUDA events, device pointers); evals/s = B / s; "
                                   "sum_n3_per_s = sum of n_b^3 over the groups / s", "workloads": {}}
    for name in ("a", "b", "c"):
        groups, jitter = workload(name)
        w = Ragged(groups, jitter)
        r = {"B": w.B, "distinct_sizes": len(w.by_size), "sum_n3": w.work,
             "sizes": {"min": int(min(len(g[0]) for g in groups)), "max": int(max(len(g[0]) for g in groups))}}
        r["ragged"] = timed(h, w.ragged, args.reps, w.B, w.work)
        ragged_out = (w.lml.cpu().numpy().copy(), w.info.cpu().numpy().copy())
        assert np.all(ragged_out[1] == 0), name
        r["per_size"] = timed(h, w.per_size, args.reps, w.B, w.work)
        r["loop"] = timed(h, w.loop, args.reps, w.B, w.work)
        loop_lml = w.lml.cpu().numpy()
        r["max_rel_diff_lml_vs_loop"] = float(np.max(np.abs(ragged_out[0] - loop_lml) / np.abs(loop_lml)))
        r["speedup_vs_loop"] = r["loop"]["ms_median"] / r["ragged"]["ms_median"]
        r["speedup_vs_per_size"] = r["per_size"]["ms_median"] / r["ragged"]["ms_median"]
        res["workloads"][name] = r
        print(name, json.dumps({k: r[k] for k in ("B", "distinct_sizes", "speedup_vs_loop", "speedup_vs_per_size")}),
              "ragged %.3f ms, per_size %.3f ms, loop %.3f ms" % (r["ragged"]["ms_median"], r["per_size"]["ms_median"],
                                                                 r["loop"]["ms_median"]), flush=True)
    b = res["workloads"]["b"]
    # workload b has one size: per_size IS the one uniform gpb200_lml_grad_batched call of the 32 groups
    b["ragged_over_uniform"] = b["ragged"]["ms_median"] / b["per_size"]["ms_median"]
    h.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"], "b_ragged_over_uniform": b["ragged_over_uniform"]}))


if __name__ == "__main__":
    main()
