"""Diagnostic: where a single-frame call spends its time (per-kernel CUDA-event times, then the un-profiled call)."""
import os, sys, time
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(REPO, "patchwork-plusplus_b200"), os.path.join(REPO, "tests")]
import pwpp_b200
from conftest import load_kitti
a = load_kitti(0)
for order in (0, 1):
    eng = pwpp_b200.Engine(device=0, num_streams=1)
    eng.set_output_order(order)
    for _ in range(5):
        eng.estimate_host([a])
    eng.set_profiling(True)
    acc = {}
    for _ in range(20):
        eng.estimate_host([a])
        for k, v in eng.stage_times_ms().items():
            acc[k] = acc.get(k, 0.0) + v * 1e3 / 20
    eng.set_profiling(False)
    for _ in range(20):
        eng.estimate_host([a])
    ts, ct = [], []
    for _ in range(200):
        t0 = time.perf_counter(); eng.estimate_host([a]); ts.append((time.perf_counter() - t0) * 1e6)
        ct.append(eng.call_times_us())
    ts.sort()
    print("order", order, "device split us (median):", {k: round(sorted(c[k] for c in ct)[100], 1) for k in ct[0]})
    print("order", order, "stage us:", {k: round(v, 1) for k, v in acc.items()}, "sum", round(sum(acc.values()), 1), "| call median us", round(ts[100], 1), "min", round(ts[0], 1), "time_us", round(eng.time_us(), 1))
    eng.close()
os.environ["PWPP_GRAPH"] = "0"
eng = pwpp_b200.Engine(device=0, num_streams=1)
for _ in range(20):
    eng.estimate_host([a])
ts = []
for _ in range(200):
    t0 = time.perf_counter(); eng.estimate_host([a]); ts.append((time.perf_counter() - t0) * 1e6)
ts.sort()
print("no graph: call median us", round(ts[100], 1), "min", round(ts[0], 1))
