"""Per-phase cycle counts of the panel kernels from an instrumented build (GPB_BUILD_TAG=trace GPB_EXTRA_NVCC=-DGPB_PANEL_TRACE
python gp_b200/build.py; GPB200_LIB=gp_b200/lib/libgpb200_trace.so python tools/panel_trace.py)."""
import sys
import numpy as np
sys.path.insert(0, ".")
from gp_b200 import capi
h = capi.Handle(0)
buf = np.zeros(2048, dtype=np.int64)
h.debug_bench_panel(0, 8, 1, 1)
assert h.lib.gpb200_debug_panel_trace(h._h, buf.ctypes.data) == 0
for name, base in (("panel warp", 512), ("helper warp 7", 0)):
    t = buf[base:base + 19 * 8].reshape(19, 8)
    print(name, "start->loaded", t[17, 0] - t[18, 0], "prologue factor", t[0, 0] - t[17, 0], "loop", t[16, 0] - t[0, 0], "writeback", t[16, 1] - t[16, 0])
    print(" step: phase1 work | barrier wait | phase2 pre-factor | factor/update | barrier wait")
    for cb in range(16):
        r = t[cb]
        if cb < 15:
            print("  %2d: %5d | %5d | %5d | %5d | %5d   (step total %d)" % (cb, r[1] - r[0], r[2] - r[1], (r[3] - r[2]) if base == 512 else 0,
                                                                    (r[4] - r[3]) if base == 512 else (r[4] - r[2]), r[5] - r[4], t[cb + 1, 0] - r[0]))
        else:
            print("  %2d: %5d | %5d" % (cb, r[1] - r[0], r[2] - r[1]))
buf[:] = 0
h2 = capi.Handle(0)
h2.debug_bench_panel(1, 8, 1, 1)   # seven row tiles: trsm_ll_kernel<1>
assert h2.lib.gpb200_debug_panel_trace(h2._h, buf.ctypes.data) == 0
t = buf[1024:1024 + 19 * 8].reshape(19, 8)
print("trsm warp 0: load+setup", t[17, 0] - t[18, 0], "loop", t[16, 0] - t[0, 0])
for cb in range(16):
    print("  %2d: dmma update %5d | solve %5d" % (cb, t[cb, 1] - t[cb, 0], t[cb, 2] - t[cb, 1]))

# the fused POTRF + TRSM launch: diagonal CTA (block 0), last TRSM CTA (compute warp 0 and the loader warp); clocks are per SM
buf[:] = 0
h3 = capi.Handle(0)
print("fused launch ms", h3.debug_bench_panel(3, 8, 1, 1))
assert h3.lib.gpb200_debug_panel_trace(h3._h, buf.ctypes.data) == 0
t = buf[512:512 + 19 * 8].reshape(19, 8)
print("fused: diagonal CTA panel warp: start->loaded", t[17, 0] - t[18, 0], "loop", t[16, 0] - t[0, 0])
print("  step totals", [int(t[cb + 1, 0] - t[cb, 0]) for cb in range(15)])
for cb in (2, 6, 10, 14):
    r = t[cb]
    print("  %2d: phase1 %5d | barrier %5d | pre-factor %5d | factor %5d | barrier %5d" % (cb, r[1] - r[0], r[2] - r[1], r[3] - r[2], r[4] - r[3], r[5] - r[4]))
hw = buf[0:19 * 8].reshape(19, 8)
for cb in (2, 6, 10, 14):
    r = hw[cb]
    print("  helper 7 %2d: phase1 %5d | barrier %5d | update %5d | barrier %5d" % (cb, r[1] - r[0], r[2] - r[1], r[4] - r[2], r[5] - r[4]))
c = buf[1024:1024 + 19 * 8].reshape(19, 8)
l = buf[1536:1536 + 16 * 8].reshape(16, 8)
print("fused: TRSM CTA compute warp 0: prologue", c[17, 0] - c[18, 0], "loop", c[16, 0] - c[0, 0], "| loader loop", l[15, 2] - l[0, 0])
for cb in range(16):
    print("  %2d: update %5d | wait for block %5d | solve+store %5d || loader: poll %5d | copy %5d | block ready at %6d, compute arrives at %6d" % (
        cb, c[cb, 3] - c[cb, 0], c[cb, 1] - c[cb, 3], c[cb, 2] - c[cb, 1], l[cb, 1] - l[cb, 0], l[cb, 2] - l[cb, 1],
        l[cb, 2] - l[0, 0], c[cb, 3] - l[0, 0]))
