"""Posterior draws over hyper-parameter samples: the per-draw route against one batched call.

  python tools/bench_posterior_draws.py [--out DIR] [--reps 3] [--shapes pendulum,lorenz,ch2]

Per-draw route, the way the reference's loops do it (pendulum_fit.R:259-268 over sample_derivs :227-255;
lorenz.Rmd:80-107; ch2.py:36-45): three gram_outer calls, gp_condition and mvrnorm(1, ..., seed = b) for each
draw b (for the pendulum shape literally ode_gp_library.sample_derivs).  Batched route: one
gpb200_posterior_draws_batched call (Handle.posterior_draws_batched, seed stream).  Both run in host-pointer mode
on the same seeded inputs and are timed end to end (wall clock; host mode synchronises before returning).
Before timing, the posterior means of the two routes must agree to 1e-9 (relative, per item).

Shapes (n training points, m prediction points, derivative order, batch):
  pendulum  n = 512, m = 512 (s = t), order 1, B = 200   pendulum_fit.R: 100 draws x 2 states
  lorenz    n = 512, m = 1024 (separate grid), order 1, B = 500, jitter 1e-6   lorenz.Rmd: 5 step sizes x 100 draws
  ch2       n = 4, m = 1000, order 0, B = 256, sigma = 0, jitter 1e-10         ch2.py:36-45
each also at B = 1 and B = 16.  Writes DIR/posterior_draws.json with the card name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, HERE)

from gp_b200 import capi, ode_gp_library as lib  # noqa: E402

KINDS = {0: ("QQ", "QQ"), 1: ("RQ", "RR"), 2: ("TQ", "TT")}


def shape(name):
    rng = np.random.default_rng({"pendulum": 1, "lorenz": 2, "ch2": 3}[name])
    if name == "pendulum":
        t = np.linspace(0.0, 10.0, 512)
        y = np.sin(t) * np.exp(-0.1 * t) + 0.05 * rng.standard_normal(512)
        return dict(t=t, s=None, y=y, order=1, B=200, jitter=1e-8, theta=lambda B: np.column_stack(
            [rng.uniform(0.8, 1.5, B), rng.uniform(0.8, 2.0, B), rng.uniform(0.03, 0.1, B)]))
    if name == "lorenz":
        t = np.linspace(0.0, 20.0, 512)
        y = 8.0 * np.sin(0.7 * t) + np.cos(1.9 * t) + 0.1 * rng.standard_normal(512)
        return dict(t=t, s=np.linspace(0.0, 20.0, 1024), y=y, order=1, B=500, jitter=1e-6, theta=lambda B: np.column_stack(
            [rng.uniform(3.0, 8.0, B), rng.uniform(0.6, 1.2, B), rng.uniform(0.05, 0.2, B)]))
    xd = np.array([-4.0, -3.0, -1.0, 2.0])
    return dict(t=xd, s=np.linspace(-5.0, 5.0, 1000), y=np.sin(xd), order=0, B=256, jitter=1e-10,
                theta=lambda B: np.column_stack([rng.uniform(0.8, 1.2, B), rng.uniform(0.8, 1.5, B), np.zeros(B)]))


def moments(h, sh, th):
    """mu and cov of one draw by the per-draw route (three Grams + gp_condition)"""
    t, s = sh["t"], sh["t"] if sh["s"] is None else sh["s"]
    alpha, rho, sigma = th
    if sh["s"] is None and sh["order"] == 1:            # pendulum_fit.R:227-251 as the library mirrors it
        return lib.sample_derivs_moments((rho, alpha, sigma), sh["y"], t, handle=h)
    a2 = alpha * alpha
    K = h.gram_outer("QQ", t, t, rho, a2)
    Ks = h.gram_outer(KINDS[sh["order"]][0], s, t, rho, a2)
    Kss = h.gram_outer(KINDS[sh["order"]][1], s, s, rho, a2)
    return h.gp_condition(K, Ks, Kss, sh["y"], sigma * sigma, sh["jitter"])


def per_draw(h, sh, th, seed):
    if sh["s"] is None and sh["order"] == 1:            # sample_derivs(params, ynoise, ti) of pendulum_fit.R:227-255
        return lib.sample_derivs((th[1], th[0], th[2]), sh["y"], sh["t"], seed=seed, handle=h)
    mu, cov = moments(h, sh, th)
    return h.mvrnorm(1, mu, cov, seed)


def loop(h, sh, th):
    return [per_draw(h, sh, th[b], b) for b in range(th.shape[0])]


def batched(h, sh, th):
    return h.posterior_draws_batched(sh["t"], sh["y"], th, order=sh["order"], s=sh["s"], jitter=sh["jitter"], seed=0)


def timed(fn, reps):
    best, total = float("inf"), 0.0
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        best, total = min(best, dt), total + dt
    return best, total / reps


def card():
    import torch
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        out["nvidia_smi"] = q
        out["power_limit_w"] = float(q.split(",")[1].strip().split()[0])
    except Exception as e:  # the measurement stands without it, but says so
        out["power_limit_w"] = None
        out["power_limit_error"] = repr(e)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=".", help="directory for posterior_draws.json")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--shapes", default="pendulum,lorenz,ch2")
    args = ap.parse_args()
    h = capi.Handle(0)
    result = {"what": "posterior draws over hyper-parameter samples: per-draw loop vs one batched call, host pointers, "
                      "wall clock after a synchronise; draws_per_s = B / mean time", "card": card(), "runs": []}
    for name in args.shapes.split(","):
        sh = shape(name)
        n, m = sh["t"].shape[0], sh["t"].shape[0] if sh["s"] is None else sh["s"].shape[0]
        th_full = sh["theta"](sh["B"])
        for B in sorted({1, 16, sh["B"]}):
            th = th_full[:B]
            draws, mu, info = batched(h, sh, th)          # also the warm-up of both routes at this shape
            loop(h, sh, th[:1])
            assert np.all(info == 0), info
            ref = [moments(h, sh, th[b])[0] for b in range(B)]
            err = max(float(np.max(np.abs(mu[b] - ref[b])) / np.max(np.abs(ref[b]))) for b in range(B))
            assert err < 1e-9, (name, B, err)
            reps_loop = 1 if B * n * m > 16 * 512 * 1024 else args.reps
            tb_best, tb_mean = timed(lambda: batched(h, sh, th), args.reps)
            tl_best, tl_mean = timed(lambda: loop(h, sh, th), reps_loop)
            r = {"shape": name, "n": n, "m": m, "order": sh["order"], "B": B, "jitter": sh["jitter"], "mu_max_rel_diff": err,
                 "batched_s": tb_mean, "batched_best_s": tb_best, "loop_s": tl_mean, "loop_best_s": tl_best,
                 "reps_batched": args.reps, "reps_loop": reps_loop,
                 "batched_draws_per_s": B / tb_mean, "loop_draws_per_s": B / tl_mean, "speedup": tl_mean / tb_mean}
            print(json.dumps(r), flush=True)
            result["runs"].append(r)
    h.close()
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "posterior_draws.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", path, "card", result["card"])


if __name__ == "__main__":
    main()
