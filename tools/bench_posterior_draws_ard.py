"""Posterior draws over ARD hyper-parameter samples: the per-draw route against one batched call.

  python tools/bench_posterior_draws_ard.py [--out DIR] [--reps 3] [--shapes pendulum,lorenz,ard8,d1]

Per-draw route, the way a user predicts on multi-column states today: for each draw b three gram_ard calls (K, Ks,
Kss: QQard of R/kernels.R:19), gp_condition and mvrnorm(1, ..., seed = b).  Batched route: one
gpb200_posterior_draws_ard_batched call (Handle.posterior_draws_ard_batched, seed stream).  Both run in host-pointer
mode on the same seeded inputs and are timed end to end (wall clock; host mode synchronises before returning).  Before
timing, the posterior means of the two routes must agree to 1e-9 (relative, per item).

Shapes (D input columns, n training points, m prediction points, batch); states as in create_p_dotXnS
(R/ode_gp_library.R:43-93):
  pendulum  D = 2, n = 512, Xs = X (m = 512), B = 200
  lorenz    D = 3, n = 512, separate Xs, m = 1024, B = 500, jitter 1e-6
  ard8      D = 8, n = 1024, separate Xs, m = 1024, B = 64
  d1        D = 1 at the lorenz n, m and B: the batched ARD call against gpb200_posterior_draws_batched at order 0
each also at B = 1 and B = 16.  Writes DIR/posterior_draws_ard.json with the card name and power limit."""
import argparse
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, HERE)

from gp_b200 import capi  # noqa: E402
from tools.bench_posterior_draws import card, timed  # noqa: E402


def _states(rng, n, D):
    """n states of a D-dimensional trajectory: smooth curves through the unit cube, plus a little noise"""
    t = np.linspace(0.0, 10.0, n)
    return np.column_stack([np.sin((0.4 + 0.3 * d) * t + d) for d in range(D)]) + 0.01 * rng.standard_normal((n, D))


def shape(name):
    rng = np.random.default_rng({"pendulum": 1, "lorenz": 2, "ard8": 3, "d1": 4}[name])
    D, n, m, B, jitter, separate = {"pendulum": (2, 512, 512, 200, 1e-8, False), "lorenz": (3, 512, 1024, 500, 1e-6, True),
                                    "ard8": (8, 1024, 1024, 64, 1e-6, True), "d1": (1, 512, 1024, 500, 1e-6, True)}[name]
    X = _states(rng, n, D)
    Xs = _states(rng, m, D) + 0.05 if separate else None
    y = np.sin(X).sum(axis=1) + 0.05 * rng.standard_normal(n)
    return dict(X=X, Xs=Xs, y=y, D=D, n=n, m=m, B=B, jitter=jitter, theta=lambda B: np.column_stack(
        [rng.uniform(0.8, 1.5, B), rng.uniform(0.5, 1.5, (B, D)), rng.uniform(0.05, 0.2, B)]))


def moments(h, sh, th):
    """mu and cov of one draw by the per-draw route (three ARD Grams + gp_condition)"""
    X = sh["X"]
    Xs = X if sh["Xs"] is None else sh["Xs"]
    alpha, rho, sigma = th[0], th[1:-1], th[-1]
    K = h.gram_ard(X, X, alpha, rho)
    Ks = h.gram_ard(Xs, X, alpha, rho)
    Kss = h.gram_ard(Xs, Xs, alpha, rho)
    return h.gp_condition(K, Ks, Kss, sh["y"], sigma * sigma, sh["jitter"])


def loop(h, sh, th):
    out = []
    for b in range(th.shape[0]):
        mu, cov = moments(h, sh, th[b])
        out.append(h.mvrnorm(1, mu, cov, b))
    return out


def batched(h, sh, th):
    return h.posterior_draws_ard_batched(sh["X"], sh["y"], th, Xs=sh["Xs"], jitter=sh["jitter"], seed=0)


def batched_se(h, sh, th):
    return h.posterior_draws_batched(sh["X"][:, 0], sh["y"], th, order=0, s=None if sh["Xs"] is None else sh["Xs"][:, 0],
                                     jitter=sh["jitter"], seed=0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=".", help="directory for posterior_draws_ard.json")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--shapes", default="pendulum,lorenz,ard8,d1")
    args = ap.parse_args()
    h = capi.Handle(0)
    result = {"what": "posterior draws over ARD hyper-parameter samples: per-draw loop (or, for d1, the 1-D SE call at "
                      "order 0) vs one batched call, host pointers, wall clock after a synchronise; draws_per_s = B / mean "
                      "time", "card": card(), "runs": []}
    for name in args.shapes.split(","):
        sh = shape(name)
        n, m = sh["n"], sh["m"]
        th_full = sh["theta"](sh["B"])
        for B in sorted({1, 16, sh["B"]}):
            th = th_full[:B]
            draws, mu, info = batched(h, sh, th)          # also the warm-up of both routes at this shape
            assert np.all(info == 0), info
            if name == "d1":
                other = lambda: batched_se(h, sh, th)
                d0, ref, i0 = other()
                assert np.all(i0 == 0), i0
                reps_other = args.reps
            else:
                other = lambda: loop(h, sh, th)
                loop(h, sh, th[:1])
                ref = [moments(h, sh, th[b])[0] for b in range(B)]
                reps_other = 1 if B * n * m > 16 * 512 * 1024 else args.reps
            err = max(float(np.max(np.abs(mu[b] - ref[b])) / np.max(np.abs(ref[b]))) for b in range(B))
            assert err < 1e-9, (name, B, err)
            tb_best, tb_mean = timed(lambda: batched(h, sh, th), args.reps)
            to_best, to_mean = timed(other, reps_other)
            r = {"shape": name, "D": sh["D"], "n": n, "m": m, "B": B, "jitter": sh["jitter"], "Xs": "X" if sh["Xs"] is None else "separate",
                 "mu_max_rel_diff": err, "batched_s": tb_mean, "batched_best_s": tb_best, "reps_batched": args.reps,
                 "batched_draws_per_s": B / tb_mean}
            if name == "d1":
                r.update({"se_order0_s": to_mean, "se_order0_best_s": to_best, "reps_se": reps_other,
                          "ard_over_se": tb_mean / to_mean, "ard_over_se_best": tb_best / to_best})
            else:
                r.update({"loop_s": to_mean, "loop_best_s": to_best, "reps_loop": reps_other, "loop_draws_per_s": B / to_mean,
                          "speedup": to_mean / tb_mean})
            print(json.dumps(r), flush=True)
            result["runs"].append(r)
    h.close()
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "posterior_draws_ard.json")
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", path, "card", result["card"])


if __name__ == "__main__":
    main()
