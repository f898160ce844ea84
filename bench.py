#!/usr/bin/env python
"""bench.py — frames/sec of the estimateGround() hot path on synthetic KITTI-64-shaped scans.

  python bench.py [--gpus N] [--steps K] [--warmup W]            our CUDA path (one process per GPU under torchrun)
  python bench.py --impl reference [...]                         the reference's own CPU estimateGround on the host cores
  python bench.py [...] --dump-outputs DIR                       also write what the last timed step computed to DIR/*.npy

Workload (BASELINE.json configs[2], the configuration the metric is quoted on): a batch of 1024 synthetic KITTI-64
frames (~120k points each) per GPU, each frame on its own FRESH stream state. A "step" is one pass of the whole path
over that batch. Frames shard across GPUs by global frame index with no data-path collective (weak scaling).

value   : frames/s with the batch resident in HBM when the timed region starts (CUDA events, max over ranks)
e2e     : the same metric through the C-ABI host entry point with page-locked HOST buffers: host->device copy of the
          batch and device->host read of all index lists inside the timed region
roofline: per kernel, 20 B/point (16 B cloud read + 4 B index write, SURVEY.md §8d) x the points that kernel's own work queue holds /
          its mean CUDA-event time (roofline.per_kernel; the top-level fields are the slowest kernel's); whole_path_frac = 20 B x
          all points / step time is the primary figure
cpu_baseline / --impl reference: the reference's patchworkpp.cpp (compiled against oracle/eigen_shim into
          oracle/_ref/libpwref.so, unmodified control flow) on all host cores, one instance per frame.
extra records (skipped with --no-extras): streaming (S streams x T consecutive frames, state carried), dense1m (BASELINE config 5
          shape), reference_order (the timed batch with the reference's emission order inside a patch), kitti_scans (the six recorded
          scans of tests/golden/ cycled to the batch size), latency_us (config 2: one frame per call through the drop-in C++ class),
          parity_vs_reference (labels of the timed result against the reference's own code on the same arrays).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(REPO, "patchwork-plusplus_b200")
for p in (PKG, os.path.join(PKG, "lib"), os.path.join(REPO, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

SEED = 20260922
METRIC = "frames/sec (120k-pt KITTI cloud)"
UNIT = "frames/s"
ALGO_BYTES_PER_POINT = 20  # SURVEY.md §8(d): 16 B/pt compulsory read of the N x 4 f32 cloud + 4 B/pt int32 index write
DUMP_SAMPLE_FRAMES = 32          # --dump-outputs: index lists of at most this many frames,
DUMP_LIST_BYTES = 48 << 20       # and at most this many bytes of them (everything dumped stays under 64 MB)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames-per-gpu", type=int, default=1024)
    ap.add_argument("--sensor", default="kitti64", choices=["kitti64", "ouster128", "dense1m"])
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--ref-frames-per-step", type=int, default=0, help="--impl reference: frames per step (0 = 8 x cores)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--streaming", default="64x16", help="streaming mode 'SxT': S sensor streams x T consecutive frames each, T batched calls with the temporal state carried (SURVEY.md 8d config 3); reported under the key 'streaming' ('' = skip)")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra records: streaming, dense1m (BASELINE config 5 shape, 32 frames per GPU), latency_us (config 2), parity_vs_reference")
    ap.add_argument("--dense-frames", type=int, default=32, help="frames per GPU of the dense1m sub-record")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to DIR/<name>.npy "
                    "(float64 / float32): per-frame counts, heights and a fixed, seeded sample of frames' index lists, centers and normals")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    return a


def merge_front_stages(stage_ms):
    """The cluster front end (k_front_cluster, the default) is ONE launch that the C-ABI reports in the first of its three
    front-end stage slots (k_bin_hist, k_bin_scan, k_scatter: the PWPP_FRONT=0 kernels); the other two slots then only hold
    the gap between two event records. Report it under its own name so that no per-kernel figure is computed for an empty slot."""
    h, sc, st = (stage_ms.get(k, 0.0) for k in ("k_bin_hist", "k_bin_scan", "k_scatter"))
    if h > 0 and sc < 0.02 * h and st < 0.02 * h:
        out = {"k_front": h + sc + st}
        out.update({k: v for k, v in stage_ms.items() if k not in ("k_bin_hist", "k_bin_scan", "k_scatter")})
        return out
    return stage_ms


# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            c = [x.strip() for x in r.split(",")]
            if len(c) < 7:
                continue
            try:
                sm.append(float(c[0])); mx.append(float(c[1]))
            except ValueError:
                continue
            for nme, v in zip(names, c[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


class NvmlSampler:
    """SM clock and clock-event reasons through NVML every ~5 ms with host timestamps, so that the samples INSIDE the timed
    region can be told from the ones around it (nvidia-smi's 200 ms loop catches at most one of a 60 ms region).
    Best effort: any failure leaves `rows` empty and the nvidia-smi sampler's numbers are used."""

    def __init__(self, index):
        self.rows = []          # (perf_counter, sm_mhz, reasons bit mask)
        self.max_mhz = None
        self._stop = False
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def start(self):
        if self.nv is None:
            return
        self._t = threading.Thread(target=self._loop, daemon=True)
        self._t.start()

    def _loop(self):
        nv = self.nv
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
        while not self._stop:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                rs = int(get_reasons(self.h)) if get_reasons else 0
                self.rows.append((time.perf_counter(), mhz, rs))
            except Exception:
                return
            time.sleep(0.005)

    def stop(self, t0, t1):
        """Summary of the samples taken in [t0, t1] (perf_counter), or None when there is none."""
        self._stop = True
        if self._t:
            self._t.join(timeout=1)
        inside = [r for r in self.rows if t0 <= r[0] <= t1]
        if not inside:
            return None
        nv = self.nv
        sm = sorted(r[1] for r in inside)
        bits = 0
        for r in inside:
            bits |= r[2]
        names = [("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_mhz, "reasons": [n for n, b in names if bits & b], "samples": len(inside),
                "source": "NVML, 5 ms period, samples inside the timed region only"}


def measured_peak_gbs():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def cpu_reference_throughput(frames, seconds_budget, max_frames=None, threads=None, cycle=False):
    """The reference's own estimateGround (oracle/_ref/libpwref.so) on `threads` host threads, a fresh instance per
    frame like config 3. ctypes releases the GIL during the foreign call, so Python threads scale across cores."""
    sys.path.insert(0, os.path.join(REPO, "oracle"))
    import oracle_py as O
    kind = "reference"
    try:
        O.Reference().close()
        mk = lambda: O.Reference(stable_sort=False)  # noqa: E731
    except Exception:
        kind = "port"
        mk = lambda: O.Oracle(arith=O.ARITH_REF32)  # noqa: E731
    T = threads or os.cpu_count() or 1
    T = max(1, min(T, len(frames)))
    done = [0] * T
    stop_at = time.perf_counter() + seconds_budget
    lim = len(frames) if max_frames is None else min(max_frames, len(frames))

    def work(t):
        i = t
        # every thread walks its share of the sample; when a time budget is given the sample is cycled until the
        # budget is used up (the GPU box has >100 cores: one pass over a few hundred frames lasts < 1 s)
        while time.perf_counter() < stop_at:
            if i >= lim:
                if not cycle:
                    break
                i = t
            r = mk()
            r.estimate(frames[i])
            r.getGroundIndices(); r.getNongroundIndices()
            r.close()
            done[t] += 1
            i += T

    t0 = time.perf_counter()
    th = [threading.Thread(target=work, args=(t,)) for t in range(T)]
    [x.start() for x in th]
    [x.join() for x in th]
    dt = time.perf_counter() - t0
    n = sum(done)
    return {"value": n / dt if dt > 0 else 0.0, "unit": UNIT, "cores": T, "kind": kind,
            "sample": f"{n} estimateGround calls over {min(lim, len(frames))} frames of the same synthetic batch, fresh instance per call, {dt:.1f} s wall on {T} threads"}, n, dt


def dump_outputs(eng, nframes, out_dir):
    """What the engine's last call computed, read back through the C-ABI like a caller would: per frame the ground / non-ground
    counts, the number of patches and the sensor height; for a sample of frames drawn with the bench seed (the same frames from
    run to run) their ground and non-ground index lists in emission order, concatenated in ascending frame order, and the patch
    centers and normals. Integers are written as float64 (exact), the engine's float32 outputs as float32."""
    import numpy as np
    counts = {name: np.array([fn(f) for f in range(nframes)], np.float64) for name, fn in
              (("num_ground", eng.num_ground), ("num_nonground", eng.num_nonground), ("num_patches", eng.num_patches), ("height", eng.height))}
    sample, list_bytes = [], 0
    for f in np.random.default_rng(SEED).permutation(nframes)[:DUMP_SAMPLE_FRAMES]:
        nb = 8 * int(counts["num_ground"][f] + counts["num_nonground"][f])
        if sample and list_bytes + nb > DUMP_LIST_BYTES:
            break
        sample.append(int(f))
        list_bytes += nb
    sample.sort()
    out = dict(counts, sample_frames=np.array(sample, np.float64))
    for name, fn, dtype in (("ground_indices", eng.ground_indices, np.float64), ("nonground_indices", eng.nonground_indices, np.float64),
                            ("centers", eng.centers, np.float32), ("normals", eng.normals, np.float32)):
        out[name] = np.concatenate([fn(f) for f in sample]).astype(dtype)
    total = sum(a.nbytes for a in out.values())
    assert total <= 64 << 20, f"--dump-outputs: {total} bytes"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # the CPU arm runs on rank 0 only
    import synth
    T = os.cpu_count() or 1
    per_step = args.ref_frames_per_step or 8 * T
    per_step = min(per_step, args.frames_per_gpu)
    dev = "cpu"
    try:
        import torch
        if torch.cuda.is_available():
            dev = "cuda"
    except Exception:
        pass
    frames = [synth.make_frame(SEED, f, args.sensor, dev).cpu().numpy() for f in range(per_step)]
    mean_pts = sum(len(f) for f in frames) / len(frames)
    for _ in range(args.warmup):
        cpu_reference_throughput(frames, 1e9)
    t0 = time.perf_counter()
    total = 0
    info = None
    for _ in range(args.steps):
        info, n, _dt = cpu_reference_throughput(frames, 1e9)
        total += n
    dt = time.perf_counter() - t0
    val = total / dt
    info["value"] = val
    info["sample"] = f"{per_step} frames per step x {args.steps} steps, fresh instance per frame, {T} threads"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": f"batch of synthetic {args.sensor} frames (~{mean_pts / 1e3:.0f}k pts), fresh state per frame; CPU sample of {per_step} frames/step",
                   "frames_per_step": per_step, "mean_points": mean_pts},
        "cpu_baseline": info,
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def run_ours(args):
    import numpy as np
    import torch
    import pwpp_b200
    import synth

    import pwpp_dist
    rank, world, local = pwpp_dist.env_rank_world()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    # one process per GPU: pin this process (and the page-locked buffers it allocates from here on) to the GPU's NUMA node
    full_affinity = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    numa_node = pwpp_b200.bind_host_to_device(local)
    dist = pwpp_dist.Dist(backend="nccl")   # rendezvous + barriers + max-over-ranks only; no data-path collective
    barrier = dist.barrier

    F = args.frames_per_gpu
    dev = torch.device("cuda", local)
    shard = pwpp_dist.weak_shard(F, rank, world)   # frames rank*F .. rank*F+F-1 of the global batch
    pts, offs = synth.make_batch(SEED, shard.start, F, args.sensor, dev)
    offs_np = offs.numpy()
    total_pts = int(offs_np[-1])
    mean_pts = total_pts / F
    eng = pwpp_b200.Engine(device=local, num_streams=F, max_points_per_frame=int(np.diff(offs_np).max()))
    # All timing uses CUDA events ON THE STREAM THE KERNELS RUN ON: an explicit torch stream whose handle is passed to
    # pwpp_estimate_device (the legacy default stream has handle 0, which the C-ABI reads as "use the ctx's own
    # stream" - torch events would then not see the kernels at all).
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0

    def step():
        eng.reset()  # every frame on a fresh stream state (config 3); stream-ordered, no host sync
        eng.estimate_device(pts.data_ptr(), offs_np, True, stream)

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    launches0 = eng.launch_count()
    clocks = ClockSampler(local)
    nvml = NvmlSampler(local)
    barrier(); torch.cuda.synchronize()
    clocks.start(); nvml.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_region0 = time.perf_counter()
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    torch.cuda.synchronize()
    t_region1 = time.perf_counter()
    barrier()
    clk = clocks.stop()
    try:
        clk_nvml = nvml.stop(t_region0, t_region1)
    except Exception:
        clk_nvml = None
    if clk_nvml is not None:
        clk_nvml["nvidia_smi"] = clk      # the 200 ms nvidia-smi loop next to it, for reference
        clk = clk_nvml
    ms = ev0.elapsed_time(ev1)
    launches = eng.launch_count() - launches0
    if args.dump_outputs:
        dump_outputs(eng, F, args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, f"rank{rank}"))
    # per-kernel device times: the same steps once more with CUDA events around every kernel (the five fit kernels,
    # which otherwise overlap on side streams, are serialised for this)
    eng.set_profiling(True)
    stage_acc = {}
    for _ in range(args.steps):
        step()
        for k, v in eng.stage_times_ms().items():
            stage_acc[k] = stage_acc.get(k, 0.0) + v
    torch.cuda.synchronize()
    eng.set_profiling(False)
    ms_ranks = dist.gather_floats(ms) if hasattr(dist, 'gather_floats') else [ms]
    ms = dist.max_over_ranks(ms)
    value = world * F * args.steps / (ms / 1e3)

    # size-independent sanity of the timed result: every frame's lists partition its points
    ng = [eng.num_ground(f) + eng.num_nonground(f) for f in range(0, F, max(1, F // 16))]
    assert all(a == int(offs_np[f + 1] - offs_np[f]) for a, f in zip(ng, range(0, F, max(1, F // 16)))), "partition invariant violated"

    # ---- roofline: every kernel against the points IT processes (20 B/point algorithmic) ----
    # the front end, k_gle and k_emit see every point; a fit kernel only the points of the patches in its size class
    # (class limits of csrc/pwpp_fit.cuh; patch sizes read back from a sample of frames and scaled to the batch)
    stage_ms = {k: v / args.steps for k, v in stage_acc.items()}
    stage_ms = merge_front_stages(stage_ms)
    peak, peak_src = measured_peak_gbs()
    sample_f = list(range(0, F, max(1, F // 64)))
    cls_pts = {"k_fit_S": 0, "k_fit_M": 0, "k_fit_L1": 0, "k_fit_L2": 0, "k_fit_L3": 0, "k_fit_X": 0}
    samp_pts = 0
    for f in sample_f:
        br = np.frombuffer(eng.bin_results(f), dtype=np.dtype([("d", np.float64, 10), ("n", np.int32), ("ng", np.int32), ("verdict", np.int32), ("fitted", np.int32)]))
        nfit = br["n"][br["fitted"] != 0].astype(np.int64)
        samp_pts += int(offs_np[f + 1] - offs_np[f])
        for name, lo, hi in (("k_fit_S", 0, 64), ("k_fit_M", 64, 512), ("k_fit_L1", 512, 2048), ("k_fit_L2", 2048, 4096), ("k_fit_L3", 4096, 8192), ("k_fit_X", 8192, 1 << 30)):
            cls_pts[name] += int(nfit[(nfit > lo) & (nfit <= hi)].sum())
    scale = total_pts / max(samp_pts, 1)
    per_kernel = {}
    for k, t in stage_ms.items():
        pts_k = cls_pts[k] * scale if k in cls_pts else float(total_pts)
        gbs = ALGO_BYTES_PER_POINT * pts_k / max(t, 1e-9) / 1e6
        per_kernel[k] = {"ms": t, "points": int(pts_k), "achieved_gbs": gbs, "frac": gbs / peak}
    top = max(stage_ms, key=stage_ms.get)
    traffic = None
    tpath = os.path.join(REPO, "profiles", "traffic.json")  # dram bytes per launch from the committed ncu --set full capture
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            if top in tj and tj[top].get("frames") and tj[top].get("dram_bytes"):
                traffic = tj[top]["dram_bytes"] / tj[top]["frames"] * F
        except Exception:
            pass
    whole = (ALGO_BYTES_PER_POINT * total_pts / (ms / args.steps / 1e3) / 1e9) / peak
    roofline = {"bound": "hbm", "kernel": top, "achieved": per_kernel[top]["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": per_kernel[top]["frac"],
                "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": ALGO_BYTES_PER_POINT * per_kernel[top]["points"],
                "accounting": "achieved = 20 B x the points the kernel's own work queue holds / its mean CUDA-event time; whole_path_frac = 20 B x all points / step time (the primary figure)",
                "whole_path_frac": whole, "whole_path_achieved_gbs": whole * peak, "per_kernel": per_kernel, "stage_ms": stage_ms,
                "stage_ms_note": "mean over K extra steps with CUDA events around every kernel (fit kernels serialised); the timed region itself runs without them"}

    # ---- end to end through the host entry point of the C-ABI (page-locked host buffers) ----
    e2e = None
    if not args.no_e2e:
        host = torch.empty((total_pts, 4), dtype=torch.float32, pin_memory=True)
        host.copy_(pts)
        torch.cuda.synchronize()
        base = host.data_ptr()
        ptrs = [base + int(offs_np[f]) * 16 for f in range(F)]
        ns = [int(offs_np[f + 1] - offs_np[f]) for f in range(F)]
        sink = 0

        def e2e_step():
            nonlocal sink
            eng.reset()
            eng.estimate_host_strided(ptrs, ns, 4, 4, 1)      # H2D of the batch + all kernels + D2H of every frame's lists into the page-locked result buffer
            idx, ng, off = eng.host_index_lists()              # zero-copy view of all 2 x F lists (pwpp_host_results)
            sink += int(idx[0]) + int(ng[F - 1])
        e2e_step()
        barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            e2e_step()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        dt = dist.max_over_ranks(dt)
        # what the per-frame copying getters of the reference surface add on top (2 x F host memcpys out of the result buffer)
        g_bufs = [np.empty(eng.num_ground(f), np.int32) for f in range(F)]
        n_bufs = [np.empty(eng.num_nonground(f), np.int32) for f in range(F)]
        tc = time.perf_counter()
        for f in range(F):
            if g_bufs[f].size: eng.lib.pwpp_copy_ground_indices(eng._h, f, g_bufs[f].ctypes.data)
            if n_bufs[f].size: eng.lib.pwpp_copy_nonground_indices(eng._h, f, n_bufs[f].ctypes.data)
        copy_ms = 1e3 * (time.perf_counter() - tc)
        assert sum(b.size for b in g_bufs) + sum(b.size for b in n_bufs) <= total_pts
        del g_bufs, n_bufs
        h2d = total_pts * 16 + (F + 1) * 12
        e2e = {"value": world * F * args.e2e_steps / dt, "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": total_pts * 4 + 3 * F * 4, "steps": args.e2e_steps, "ms_per_step": 1e3 * dt / args.e2e_steps,
               "h2d_gbs_per_rank": h2d / (dt / args.e2e_steps) / 1e9, "numa_node": numa_node,
               "copying_getters_ms": copy_ms,
               "api": "pwpp_estimate_host + pwpp_host_results (zero-copy view of all index lists in the page-locked result buffer); copying_getters_ms = the 2 x F pwpp_copy_*_indices calls a caller that wants private copies pays on top (host memcpy, not in value)"}

    # ---- extra records (never cost the main line; collectives stay outside the try blocks) ----
    # streaming mode: S streams x T consecutive frames, state carried from call to call (SURVEY.md 8d config 3)
    streaming, sms = None, -1.0
    if args.streaming and not args.no_extras:
        try:
            S, T = (int(x) for x in args.streaming.lower().split("x"))
            assert 1 <= S and 1 <= T and S * T <= F, "needs S*T <= --frames-per-gpu"
            seng = pwpp_b200.Engine(device=local, num_streams=S, max_points_per_frame=int(np.diff(offs_np).max()))
            calls = [(int(offs_np[t * S]), (offs_np[t * S:(t + 1) * S + 1] - offs_np[t * S]).copy()) for t in range(T)]

            def sequence():
                seng.reset()
                for first, o in calls:   # call t: frame t of every stream; stream order serialises consecutive frames
                    seng.estimate_device(pts.data_ptr() + first * 16, o, True, stream)
            sequence(); torch.cuda.synchronize()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for _ in range(3):
                sequence()
            s1.record(); torch.cuda.synchronize()
            sms = s0.elapsed_time(s1) / 3
            seng.close()
        except Exception as ex:
            streaming = {"error": repr(ex)[:200]}
        sms = dist.max_over_ranks(sms)
        if streaming is None and sms > 0:
            streaming = {"streams": S, "frames_per_stream": T, "ms_per_sequence": sms, "value": world * S * T / (sms / 1e3), "unit": UNIT,
                         "ms_per_call": sms / T, "note": "T batched calls of S frames per GPU, adaptive state carried between calls"}

    # dense sensor (BASELINE config 5 shape: ~1.2 M points per frame), --dense-frames frames per GPU, device-resident
    dense, dms, dstage = None, -1.0, None
    if args.sensor == "kitti64" and not args.no_extras and args.dense_frames > 0:
        dmean = 0.0
        try:
            DF = args.dense_frames
            dshard = pwpp_dist.weak_shard(DF, rank, world)
            dpts, doffs = synth.make_batch(SEED, dshard.start, DF, "dense1m", dev)
            doffs_np = doffs.numpy()
            dmean = float(doffs_np[-1]) / DF
            deng = pwpp_b200.Engine(device=local, num_streams=DF, max_points_per_frame=int(np.diff(doffs_np).max()))

            def dstep():
                deng.reset(); deng.estimate_device(dpts.data_ptr(), doffs_np, True, stream)
            for _ in range(3):
                dstep()
            torch.cuda.synchronize()
            d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            d0.record()
            for _ in range(5):
                dstep()
            d1.record(); torch.cuda.synchronize()
            dms = d0.elapsed_time(d1) / 5
            deng.set_profiling(True); dstep(); dstage = merge_front_stages(deng.stage_times_ms()); deng.set_profiling(False)
            assert deng.num_ground(0) + deng.num_nonground(0) == int(doffs_np[1] - doffs_np[0])
            deng.close(); del dpts
        except Exception as ex:
            dense = {"error": repr(ex)[:200]}
        dms = dist.max_over_ranks(dms)
        if dense is None and dms > 0:
            dense = {"frames_per_gpu": DF, "mean_points": dmean, "ms_per_step": dms, "value": world * DF / (dms / 1e3), "unit": UNIT,
                     "points_per_s": world * DF * dmean / (dms / 1e3), "whole_path_frac": (ALGO_BYTES_PER_POINT * DF * dmean / (dms / 1e3) / 1e9) / peak,
                     "stage_ms": dstage, "workload": f"batch={DF} synthetic dense1m frames per GPU (Ouster-128 layout x 16384 azimuth steps), fresh state per frame, device-resident"}

    # the same batch with the reference's emission order inside every patch (pwpp_set_output_order(1): what the drop-in
    # C++ class / pypatchworkpp select; the main line runs the native bin-major, ascending-index order)
    ordered, oms = None, -1.0
    if not args.no_extras:
        try:
            eng.set_output_order(1)
            for _ in range(2):
                step()
            torch.cuda.synchronize()
            o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            o0.record()
            for _ in range(5):
                step()
            o1.record(); torch.cuda.synchronize()
            oms = o0.elapsed_time(o1) / 5
            eng.set_output_order(0)
            step(); torch.cuda.synchronize()   # leave the native-order result in place for the parity record below
        except Exception as ex:
            ordered = {"error": repr(ex)[:200]}
        oms = dist.max_over_ranks(oms)
        if ordered is None and oms > 0:
            ordered = {"ms_per_step": oms, "value": world * F / (oms / 1e3), "unit": UNIT,
                       "note": "k_order on: ground part of every patch in ascending z, then the R-VPF removals per iteration and the final rejects, each in ascending z (S:199, S:264-284)"}

    # real scans: the six KITTI fixture scans of tests/golden/ cycled to a batch of F frames (fresh state per frame, device-resident,
    # native emission order): the number to expect on recorded data. The synthetic generator differs from KITTI in both directions
    # (denser near the sensor and larger bins, but fewer points per frame and less vertical structure: tests/test_generator.py)
    real, rms = None, -1.0
    if not args.no_extras and args.sensor == "kitti64":
        try:
            from conftest import load_kitti
            scans = [torch.from_numpy(load_kitti(i)) for i in range(6)]
            sizes = [int(scans[f % len(scans)].shape[0]) for f in range(F)]
            roffs_np = np.zeros(F + 1, np.int64); roffs_np[1:] = np.cumsum(sizes)
            dscans = [x.to(dev) for x in scans]
            rpts = torch.cat([dscans[f % len(scans)] for f in range(F)], dim=0).contiguous()
            reng = pwpp_b200.Engine(device=local, num_streams=F, max_points_per_frame=max(sizes))

            def rstep():
                reng.reset(); reng.estimate_device(rpts.data_ptr(), roffs_np, True, stream)
            for _ in range(3):
                rstep()
            torch.cuda.synchronize()
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            r0.record()
            for _ in range(5):
                rstep()
            r1.record(); torch.cuda.synchronize()
            rms = r0.elapsed_time(r1) / 5
            reng.set_profiling(True); rstep(); rstage = merge_front_stages(reng.stage_times_ms()); reng.set_profiling(False)
            assert reng.num_ground(7) + reng.num_nonground(7) == sizes[7]
            rground = float(np.mean([reng.num_ground(f) / sizes[f] for f in range(6)]))
            reng.close(); del rpts, dscans
        except Exception as ex:
            real = {"error": repr(ex)[:200]}
        rms = dist.max_over_ranks(rms)
        if real is None and rms > 0:
            real = {"frames_per_gpu": F, "mean_points": float(roffs_np[-1]) / F, "ms_per_step": rms, "value": world * F / (rms / 1e3), "unit": UNIT,
                    "ground_fraction": rground, "whole_path_frac": (ALGO_BYTES_PER_POINT * float(roffs_np[-1]) / (rms / 1e3) / 1e9) / peak, "stage_ms": rstage,
                    "workload": f"batch={F}: the six recorded KITTI scans of tests/golden/ cycled, fresh state per frame, device-resident"}

    # single-frame latency of the drop-in C++ class (BASELINE config 2): examples/pwpp_latency.cpp on the first fixture scan
    latency = None
    if rank == 0 and not args.no_extras:
        try:
            exe = os.path.join(PKG, "lib", "pwpp_latency")
            if os.path.exists(exe):
                import tempfile
                from conftest import load_kitti
                scan = load_kitti(0)
                with tempfile.NamedTemporaryFile(suffix=".bin") as tf:
                    scan.tofile(tf.name)
                    env = dict(os.environ, CUDA_VISIBLE_DEVICES=str(local))
                    out = subprocess.run([exe, tf.name, "300", "30"], capture_output=True, text=True, timeout=120, env=env).stdout
                latency = json.loads([l for l in out.splitlines() if l.startswith("{")][-1])
                latency["what"] = "PatchWorkpp::estimateGround + getGroundIndices + getNongroundIndices on kitti_000000 (124,668 points), host clock around the call sequence, median of 300 calls after 30 warm-up calls; H2D and D2H inside"
        except Exception as ex:
            latency = {"error": repr(ex)[:200]}

    # ---- CPU baseline on the host cores of this box (rank 0 only) ----
    cpu, parity = None, None
    if rank == 0 and not args.no_cpu_baseline:
        T = os.cpu_count() or 1
        nsample = min(F, max(T * 4, 64))
        frames = [pts[int(offs_np[f]):int(offs_np[f + 1])].cpu().numpy() for f in range(nsample)]
        if full_affinity is not None:   # the GPU legs pinned this process to the GPU's NUMA node: the reference gets every host core back
            try:
                os.sched_setaffinity(0, full_affinity)
            except OSError:
                pass
        cpu, _, _ = cpu_reference_throughput(frames, args.cpu_seconds, cycle=True)
        if not args.no_extras:
            # labels of the timed result against the reference's own code on the same arrays (first 64 frames of the batch)
            try:
                import oracle_py as O
                labels = mism = 0
                for f in range(min(64, nsample)):
                    r = O.Reference(stable_sort=False); r.estimate(frames[f]); g_r = r.getGroundIndices(); r.close()
                    mr = np.zeros(len(frames[f]), bool); mr[g_r] = True
                    me = np.zeros(len(frames[f]), bool); me[eng.ground_indices(f)] = True
                    labels += len(frames[f]); mism += int((mr != me).sum())
                parity = {"frames": min(64, nsample), "labels": labels, "mismatches": mism,
                          "note": "ground / non-ground label of every point vs oracle/_ref/libpwref.so (the reference's patchworkpp.cpp, fp32) on the same arrays; the CUDA path computes in double (DESIGN.md section 3)"}
            except Exception as ex:
                parity = {"error": repr(ex)[:200]}

    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "ms_per_step_ranks": [m / args.steps for m in ms_ranks], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": f"batch={F} synthetic {args.sensor} frames (~{mean_pts / 1e3:.0f}k pts each) per GPU, fresh stream state per frame, device-resident input",
                       "frames_per_gpu": F, "mean_points": mean_pts, "sharding": "frames by global index, no collective",
                       "l2": f"inputs larger than L2: {total_pts * 16 / 1e9:.2f} GB of points per step vs 126 MB L2"},
            "clocks": clk, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
        }
        for k, v in (("streaming", streaming), ("dense1m", dense), ("reference_order", ordered), ("kitti_scans", real), ("latency_us", latency), ("parity_vs_reference", parity)):
            if v is not None:
                out[k] = v
        print(json.dumps(out), flush=True)
    # orderly teardown: release the engine (CUDA buffers, streams) while the CUDA context is still alive
    eng.close()
    del pts
    torch.cuda.synchronize()
    dist.close()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
