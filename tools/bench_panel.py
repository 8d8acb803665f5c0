"""Times the panel kernels in isolation (gpb200_debug_bench_panel), with and without the fused POTRF + TRSM
launch, at the batch sizes of the latency path (1, 4) and of the batched headline step (256)."""
import json
import os
import subprocess
import sys

sys.path.insert(0, ".")


def run_variant():
    from gp_b200 import capi
    h = capi.Handle(0)
    out = {}
    for what, name in ((0, "potrf_tile"), (1, "trsm_tiles"), (2, "tile_inverse"), (3, "potrf+trsm")):
        for nt, batch in ((32, 1), (8, 1), (32, 2), (32, 4), (8, 32), (32, 128), (64, 1), (128, 1)):
            if what == 0 and nt != 32:
                continue
            if what != 3 and nt > 32:
                continue
            out["%s nt=%d B=%d" % (name, nt, batch)] = round(h.debug_bench_panel(what, nt, batch, 5) * 1e3, 2)
    print(json.dumps(out))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "child":
        run_variant()
        sys.exit(0)
    res = {}
    for label, env in (("round2_panel_warp", {}), ("round2_two_launches", {"GPB200_PANEL_FUSED": "0"})):
        e = dict(os.environ); e.update(env)
        r = subprocess.run([sys.executable, __file__, "child"], env=e, capture_output=True, text=True)
        if r.returncode != 0:
            res[label] = {"error": r.stderr[-2000:]}
        else:
            res[label] = json.loads(r.stdout.strip().splitlines()[-1])
    print(json.dumps(res, indent=1))
    os.makedirs("gpurun_out", exist_ok=True)
    json.dump(res, open("gpurun_out/bench_panel.json", "w"), indent=1)
