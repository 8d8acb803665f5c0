"""Envelope route against a reference tree: bench.py of both, alternated, in one process tree.

  python tools/bench_envelope.py --ref DIR [--runs 3] [--steps 10] [--warmup 3] [--out DIR]
  python tools/bench_envelope.py --sweep [--rounds 3]

Runs `bench.py --gpus 1` of this tree and of the tree at DIR (built the same way) in turn, `--runs` times each, and
prints per run the headline evals/s, the LML-only `cholesky` ms, executed_tflops and the latency block; the last run
of each dumps its outputs, and the maximum relative difference of lml and grad between the two is printed with the
card name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(tree, args, dump):
    cmd = [sys.executable, os.path.join(tree, "bench.py"), "--gpus", "1", "--steps", str(args.steps), "--warmup",
           str(args.warmup)] + (["--dump-outputs", dump] if dump else [])
    out = subprocess.run(cmd, cwd=tree, capture_output=True, text=True)
    if out.returncode:
        raise RuntimeError(out.stderr[-4000:])
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    return json.loads(line)


def summary(r):
    lat = {k: v for k, v in (r.get("latency") or {}).items() if k != "what"}
    return {"value": r.get("value"), "cholesky_ms": r.get("cholesky", {}).get("ms_per_step"),
            "executed_tflops": r.get("roofline", {}).get("executed_tflops"),
            "other_kernels_ms_per_step": r.get("roofline", {}).get("other_kernels_ms_per_step"), "latency": lat}


def synth(n, B, seed=5, rho_scale=1.0):
    rng = np.random.default_rng(seed)
    x = np.sort(rng.uniform(0.0, 0.05 * n, size=n))
    y = np.sin(x) + 0.5 * np.sin(3.1 * x) + 0.3 * rng.standard_normal(n)
    th = np.stack([np.abs(rng.standard_normal(B)) + 0.1, rng.gamma(4.0, 0.25, B) * rho_scale, rng.uniform(0.1, 0.5, B)],
                  axis=1)
    return x, y, th


def sweep(args):
    import torch
    sys.path.insert(0, HERE)
    from gp_b200 import capi
    dev = torch.device("cuda", 0)
    stream = torch.cuda.current_stream(dev)
    handles = {}
    for name, env in (("dense", {"GPB200_ENVELOPE": "0"}), ("env_inverse", {"GPB200_SINV_MINB": "1000000"}),
                      ("env_sinv", {"GPB200_SINV_MINB": "1"})):
        old = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        h = capi.Handle(0)
        for k, v in old.items():
            if v is None: del os.environ[k]
            else: os.environ[k] = v
        h.set_stream(stream.cuda_stream)
        h.set_pointer_mode(True)
        handles[name] = h
    shapes = [(n, B, 1.0) for n in (1024, 2048, 4096) for B in (1, 4, 8, 16, 32)] + [(4096, 256, 20.0)]
    res = {}
    for r in range(args.rounds):
        for n, B, rs in shapes:
            x, y, th = synth(n, B, rho_scale=rs)
            dx, dy, dth = (torch.from_numpy(a).to(dev) for a in (x, y, th))
            lml = torch.empty(B, dtype=torch.float64, device=dev)
            grad = torch.empty(B, 3, dtype=torch.float64, device=dev)
            info = torch.zeros(B, dtype=torch.int32, device=dev)
            reps = max(2, min(20, int(2000 // max(1, B * (n // 1024) ** 3))))
            for name, h in handles.items():
                for _ in range(2):
                    h.lml_grad_batched_device(n, B, dx, 0, dy, 0, dth, 0.0, True, lml, grad, info)
                torch.cuda.synchronize(dev)
                e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(reps):
                    h.lml_grad_batched_device(n, B, dx, 0, dy, 0, dth, 0.0, True, lml, grad, info)
                e1.record(stream)
                torch.cuda.synchronize(dev)
                key = "n%d_b%d%s" % (n, B, "_dense_cov" if rs != 1.0 else "")
                res.setdefault(key, {}).setdefault(name, []).append(round(e0.elapsed_time(e1) / reps, 4))
    for k, v in res.items():
        print(json.dumps({"shape": k, "ms_per_call": v}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref")
    ap.add_argument("--sweep", action="store_true")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="directory for the dumped outputs (default: a new temporary directory)")
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(json.dumps({"gpu": smi}), flush=True)
    if args.sweep:
        return sweep(args)
    if not args.ref:
        ap.error("--ref DIR or --sweep")
    if args.out is None:
        args.out = tempfile.mkdtemp(prefix="bench_envelope_")
    args.out = os.path.abspath(args.out)
    os.makedirs(args.out, exist_ok=True)
    res = {"branch": [], "ref": []}
    for i in range(args.runs):
        last = i == args.runs - 1
        for name, tree in (("ref", os.path.abspath(args.ref)), ("branch", HERE)):
            r = run(tree, args, os.path.join(args.out, name) if last else None)
            res[name].append(r)
            print(json.dumps({"tree": name, "run": i, **summary(r)}), flush=True)
    with open(os.path.join(args.out, "runs.json"), "w") as f:
        json.dump(res, f)
    d = {}
    for key in ("lml", "grad"):
        a = np.load(os.path.join(args.out, "branch", key + ".npy"))
        b = np.load(os.path.join(args.out, "ref", key + ".npy"))
        if key == "grad":
            d[key] = float(np.max(np.max(np.abs(a - b), axis=1) / np.max(np.abs(b), axis=1)))
        else:
            d[key] = float(np.max(np.abs(a - b) / np.abs(b)))
    print(json.dumps({"max_rel_diff": d}), flush=True)


if __name__ == "__main__":
    main()
