"""CPU tests of the per-group (ragged) plumbing: the sum-of-n^3 balanced split of gp_b200/sharding.py, run across two
gloo processes with the CPU oracle injected as the evaluator; the argument checks of the Python binding that happen
before the library is reached; gp_lml_grad_groups of r/shim.c through the mock of the R C API (coercion and shape
errors); and gp_lml_groups of stan/gp_lml_stan.hpp built against the mock of Stan Math and run.  The tests marked gpu
compare the R and Stan values and adjoints with the oracle."""
import os
import socket

import numpy as np
import pytest
import torch.multiprocessing as mp

from gp_b200.sharding import weighted_bounds

SIZES = [40, 7, 90, 13, 64, 5, 33, 120, 2, 71]


def test_weighted_bounds_are_contiguous_and_balance_cost():
    rng = np.random.default_rng(1)
    for trial in range(50):
        costs = rng.integers(1, 2048, size=int(rng.integers(0, 60))).astype(float) ** 3
        for world in (1, 2, 3, 8):
            spans = [weighted_bounds(costs, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == len(costs)
            for a, b in zip(spans[:-1], spans[1:]):
                assert a[1] == b[0] and a[0] <= a[1]
            if len(costs):
                share = costs.sum() / world
                for lo, hi in spans:   # each rank's cost is its share, give or take one item on each side
                    assert abs(costs[lo:hi].sum() - share) <= 2 * costs.max() + 1e-6 * share


def test_weighted_bounds_follow_cost_not_count():
    costs = [8.0 ** 3] + [1.0] * 99   # one big group and many tiny ones
    assert weighted_bounds(costs, 0, 2) == (0, 1)
    assert weighted_bounds(costs, 1, 2) == (1, 100)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _groups():
    from oracle import gp_oracle as o
    xs, ys = zip(*[o.synth_xy(n, 20 + g) for g, n in enumerate(SIZES)])
    return list(xs), list(ys), o.synth_theta(len(SIZES), 9)


def _oracle_eval(xs, ys, theta, jitter):
    from oracle import gp_oracle as o
    B = len(xs)
    lml = np.empty(B); grad = np.empty((B, 3)); info = np.zeros(B, dtype=np.int32)
    for b in range(B):
        lml[b], grad[b] = o.lml_grad(xs[b], ys[b], *theta[b], jitter=jitter)
    return lml, grad, info


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from gp_b200.sharding import lml_grad_groups_sharded
    xs, ys, th = _groups()
    seen = []

    def ev(a, b, t, j):
        seen.extend(len(v) for v in a)
        return _oracle_eval(a, b, t, j)
    lml, grad, info = lml_grad_groups_sharded(xs, ys, th, evaluator=ev)
    q.put((rank, seen, lml, grad, info))
    dist.barrier()
    dist.destroy_process_group()


def test_world_size_2_gloo_groups_match_single_process():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=120) for _ in range(2)], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    xs, ys, th = _groups()
    ref = _oracle_eval(xs, ys, th, 0.0)
    costs = [float(n) ** 3 for n in SIZES]
    for rank, seen, lml, grad, info in res:
        lo, hi = weighted_bounds(costs, rank, 2)
        assert seen == SIZES[lo:hi]            # each rank evaluated exactly its contiguous range
        assert np.array_equal(lml, ref[0]) and np.array_equal(grad, ref[1]) and np.array_equal(info, ref[2])


def test_single_process_groups_call_the_evaluator_once():
    from gp_b200.sharding import lml_grad_groups_sharded
    xs, ys, th = _groups()
    calls = []

    def ev(a, b, t, j):
        calls.append(len(a))
        return _oracle_eval(a, b, t, j)
    lml, grad, info = lml_grad_groups_sharded(xs, ys, th, evaluator=ev)
    ref = _oracle_eval(xs, ys, th, 0.0)
    assert calls == [len(SIZES)]
    assert np.array_equal(lml, ref[0]) and np.array_equal(grad, ref[1])


def test_binding_rejects_mismatched_groups_before_the_library():
    from gp_b200 import capi
    h = capi.Handle.__new__(capi.Handle)   # no device: the checks run before any library call
    h._h = None
    with pytest.raises(capi.GpB200Error, match="groups"):
        h.lml_grad_ragged([np.zeros(3)], [np.zeros(3), np.zeros(2)], [[1.0, 1.0, 0.1]])
    with pytest.raises(capi.GpB200Error, match="as many points"):
        h.lml_grad_ragged([np.zeros(3)], [np.zeros(2)], [[1.0, 1.0, 0.1]])


# ---- R: gp_lml_grad_groups of r/shim.c through the functional mock of the R C API ----

@pytest.fixture(scope="module")
def R():
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "support"))
    import mock_r
    return mock_r


def test_r_groups_entry_is_registered_and_shape_errors_are_r_errors(R):
    r = R.MockR()
    assert r.registered("gp_lml_grad_groups") > 0
    xs = [np.arange(3.0), np.arange(5.0)]
    ys = [np.zeros(3), np.zeros(5)]
    th = np.ones((3, 2))
    with pytest.raises(R.RError, match=r"length\(y_list\) = 1 must equal length\(x_list\) = 2"):
        r.call("gp_lml_grad_groups", xs, ys[:1], th, 0.0)
    with pytest.raises(R.RError, match=r"length\(y_list\[\[2\]\]\) = 4 must equal length\(x_list\[\[2\]\]\) = 5"):
        r.call("gp_lml_grad_groups", xs, [ys[0], np.zeros(4)], th, 0.0)
    with pytest.raises(R.RError, match=r"x_list\[\[1\]\] is empty"):
        r.call("gp_lml_grad_groups", [np.zeros(0), xs[1]], [np.zeros(0), ys[1]], th, 0.0)
    with pytest.raises(R.RError, match=r"theta must be a 3 x B matrix.*B = length\(x_list\) = 2 \(got 3 x 3\)"):
        r.call("gp_lml_grad_groups", xs, ys, np.ones((3, 3)), 0.0)
    with pytest.raises(R.RError, match=r"got 2 x 2"):
        r.call("gp_lml_grad_groups", xs, ys, np.ones((2, 2)), 0.0)
    with pytest.raises(R.RError, match="lists of numeric vectors"):
        r.call("gp_lml_grad_groups", np.arange(3.0), ys, th, 0.0)
    with pytest.raises(R.RError, match="must not be NULL"):
        r.call("gp_lml_grad_groups", xs, ys, None, 0.0)


def test_r_groups_coerce_integer_inputs(R):
    import torch
    r = R.MockR()
    xs = [np.arange(4, dtype=np.int32), np.arange(9, dtype=np.int32)]   # integer vectors from R are coerced to double
    ys = [np.linspace(-1, 1, 4), np.linspace(0, 1, 9)]
    th = np.array([[1, 1], [2, 1], [1, 1]], dtype=np.int32)             # an integer theta matrix too
    if not torch.cuda.is_available():
        with pytest.raises(R.RError, match="no usable B200 GPU"):   # coercion and shapes passed: only the GPU is missing
            r.call("gp_lml_grad_groups", xs, ys, th, 0.0)
        return
    from oracle import gp_oracle as o
    out = r.call("gp_lml_grad_groups", xs, ys, th, 0.0)
    assert out["grad"].shape == (3, 2) and np.all(out["info"] == 0)
    for b in range(2):
        rv, rg = o.lml_grad(xs[b].astype(float), ys[b], *th[:, b].astype(float))
        assert abs(out["lml"][b] - rv) <= 1e-9 * abs(rv)
        assert np.all(np.abs(out["grad"][:, b] - rg) <= 1e-9 * np.abs(rg) + 1e-300)


@pytest.mark.gpu
def test_r_groups_match_the_oracle(R):
    from oracle import gp_oracle as o
    r = R.MockR()
    sizes = [3, 150, 40, 300]
    xs, ys = zip(*[o.synth_xy(n, 60 + g) for g, n in enumerate(sizes)])
    th = o.synth_theta(len(sizes), 61)
    out = r.call("gp_lml_grad_groups", list(xs), list(ys), np.asfortranarray(th.T), 1e-8)
    assert out["grad"].shape == (3, len(sizes)) and np.all(out["info"] == 0)
    for b in range(len(sizes)):
        rv, rg = o.lml_grad_lapack(xs[b], ys[b], *th[b], jitter=1e-8)
        assert abs(out["lml"][b] - rv) <= 1e-9 * abs(rv)
        assert np.all(np.abs(out["grad"][:, b] - rg) <= 1e-9 * np.abs(rg))


# ---- Stan: gp_lml_groups of stan/gp_lml_stan.hpp, built against the mock of Stan Math and run (run_groups.cpp) ----

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STAN_EXE = os.path.join(ROOT, "stan", "mock", "run_stan_groups_mock")


def _stan_build():
    import subprocess
    subprocess.check_call(["bash", os.path.join(ROOT, "stan", "mock", "build_mock.sh")], stdout=subprocess.DEVNULL)
    return STAN_EXE


def _stan_inputs():
    sizes = [1, 7, 130, 300, 64]
    xs, ys, th = [], [], []
    for g, n in enumerate(sizes):
        i = np.arange(n)
        x = 0.05 * i + 0.01 * np.sin(1.7 * i + g)
        xs.append(x); ys.append(np.sin(x) + 0.3 * np.cos(5.0 * x + g))
        th.append([1.0 + 0.1 * g, 0.8 + 0.05 * g, 0.2 + 0.03 * g])
    return xs, ys, np.array(th)


def test_stan_groups_driver_builds_links_and_fails_loudly_without_a_gpu():
    import subprocess
    import torch
    exe = _stan_build()
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 1 and "no usable B200 GPU" in r.stdout


@pytest.mark.gpu
def test_stan_groups_values_and_adjoints_match_the_oracle():
    import json
    import subprocess
    from oracle import gp_oracle as o
    r = subprocess.run([_stan_build()], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    out = json.loads(r.stdout)
    xs, ys, th = _stan_inputs()
    ref = [o.lml_grad(xs[g], ys[g], *th[g]) for g in range(len(xs))]
    total = sum(v for v, _ in ref)
    adj = np.array([g for _, g in ref])
    assert abs(out["vvv"]["value"] - total) <= 1e-9 * abs(total)
    assert np.all(np.abs(np.array(out["vvv"]["adj"]) - adj) <= 1e-9 * np.abs(adj))
    assert abs(out["dvd"]["value"] - total) <= 1e-9 * abs(total)
    assert np.all(np.abs(np.array(out["dvd"]["adj_rho"]) - adj[:, 1]) <= 1e-9 * np.abs(adj[:, 1]))
    assert abs(out["ddd"]["value"] - total) <= 1e-9 * abs(total)
    assert out["domain_error_on_singular_group"] is True
