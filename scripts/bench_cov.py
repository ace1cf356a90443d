"""Covariance pass (61 R50-FPN layers @800x1344, B=8) under the three host modes."""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench
import nsgp_repre_b200 as pkg
from nsgp_repre_b200 import standin, _lib

B = int(sys.argv[1]) if len(sys.argv) > 1 else 8
if os.environ.get("STAGE_SMS"):
    pkg.CovarianceHooks.stage_sms = int(os.environ["STAGE_SMS"])
layers = bench.trace_layers(800, 1344, standin)
g = torch.Generator(device="cuda").manual_seed(0)
xs = [torch.relu(torch.randn(B, r["Cin"], r["H"], r["W"], device="cuda", generator=g)) for r in layers]
flops = sum(r["cov_flops"] for r in layers)

def run(mode, join_each):
    hooks = pkg.CovarianceHooks(torch.nn.Identity(), mode=mode)
    def one():
        for r, x in zip(layers, xs):
            hooks._accumulate_conv(x, r["name"], (r["k"],) * 2, (r["s"],) * 2, (r["p"],) * 2)
        hooks.flush()
        if join_each:
            hooks.join()
    for _ in range(2):
        one()
    hooks.join(); torch.cuda.synchronize()
    _lib.profile_read(); _lib.profile_enable(os.environ.get("NOPROF") is None)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 5
    t0 = time.perf_counter()
    e0.record()
    for _ in range(reps):
        one()
    issue = (time.perf_counter() - t0) / reps * 1e3
    hooks.join()
    e1.record(); torch.cuda.synchronize()
    host = (time.perf_counter() - t0) / reps * 1e3
    print("host issue time per pass: %.2f ms" % issue)
    _lib.profile_enable(False)
    prof = _lib.profile_read()
    ms = e0.elapsed_time(e1) / reps
    print("%-10s join_each=%d  %.2f ms/pass (host %.2f)  %.0f TF alg | gram %.2f ms (%d launches)  stage %.2f ms" %
          (mode, join_each, ms, host, flops / ms / 1e9, prof["gram"][0] / reps, prof["gram"][1] / reps,
           prof["stage"][0] / reps))

modes = sys.argv[2].split(",") if len(sys.argv) > 2 else ("immediate", "grouped", "deferred")
def timeline():
    if not os.environ.get("NSGP_TIMELINE"):
        return
    import ctypes
    n = 512
    buf = (ctypes.c_ulonglong * (2 * n))()
    kinds = (ctypes.c_int * n)()
    m = _lib.lib.nsgp_debug_timeline_read(buf, kinds, n)
    ev = [(buf[2 * i], buf[2 * i + 1], kinds[i]) for i in range(m)]
    ev = ev[-int(os.environ.get('TL_N', '15')):]
    t0 = min(e[0] for e in ev)
    names = {2: "stage", 0: "gram-generic", 10: "gram-autocorr"}
    for a, b, k in sorted(ev):
        print("   %-14s %8.3f -> %8.3f ms  (%.3f)" % (names.get(k, k), (a - t0) / 1e6, (b - t0) / 1e6, (b - a) / 1e6))

def counters():
    if not os.environ.get("NSGP_DBG_COUNTERS"):
        return
    import ctypes
    import numpy as np
    n = 148 * 8
    buf = (ctypes.c_ulonglong * n)()
    _lib.check(_lib.lib.nsgp_debug_read_counters(buf, -n), "counters")
    c = np.array(list(buf), dtype=np.float64).reshape(148, 8)
    tot = c[:, 7].mean()
    st = max(1.0, c[:, 4].mean())
    buf2 = (ctypes.c_ulonglong * n)()
    _lib.check(_lib.lib.nsgp_debug_read_counters(buf2, n), "counters")
    g = np.array(list(buf2), dtype=np.float64).reshape(148, 8)
    gt = g[:, 5].mean()
    if gt > 0:
        print("   generic kernel per-CTA cycles: mean %.0f max %.0f min %.0f | MMA warp: wait-operands %.0f%% issue %.0f%% wait-accum %.0f%% | producer: wait-stage %.0f%% issue %.0f%% | %.0f K blocks -> %.0f cycles/K-block" %
              (gt, g[:, 5].max(), g[:, 5].min(), 100 * g[:, 0].mean() / gt, 100 * g[:, 1].mean() / gt, 100 * g[:, 2].mean() / gt,
               100 * g[:, 3].mean() / gt, 100 * g[:, 4].mean() / gt, g[:, 6].mean(), gt / max(1.0, g[:, 6].mean())))
    print("   AC kernel per-CTA cycles: mean %.0f max %.0f min %.0f (%.2f ms at 1.965 GHz), %.0f cycles/row step | MMA warp: wait-A %.0f%% wait-B %.0f%% wait-epi %.0f%% issue %.0f%%" %
          (tot, c[:, 7].max(), c[:, 7].min(), tot / 1.965e6, tot / st, 100 * c[:, 0].mean() / tot, 100 * c[:, 1].mean() / tot,
           100 * c[:, 2].mean() / tot, 100 * c[:, 3].mean() / tot))

for mode in modes:
    for je in (1, 0):
        run(mode, je)
        counters()
        timeline()
