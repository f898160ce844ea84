"""bench.py's output contract, as far as it can run without a GPU: the reference arm (`--impl reference`) executes the
reference's own CPU estimateGround and must print ONE JSON line with the keys the driver reads; the product arm must
refuse to run without a CUDA device instead of falling back to anything."""
import json
import os
import subprocess
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _no_gpu():
    try:
        import torch
        return not torch.cuda.is_available()
    except Exception:
        return True


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--frames-per-gpu", "4",
                          "--ref-frames-per-step", "4"], capture_output=True, text=True, timeout=600, cwd=REPO)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["metric"].startswith("frames/sec") and j["unit"] == "frames/s" and j["higher_is_better"] is True
    assert j["value"] > 0 and j["steps"] == 1 and j["n_gpus"] == 1 and j["scaling"] == "weak" and j["vs_baseline"] is None
    assert j["cpu_baseline"]["kind"] in ("reference", "port") and j["cpu_baseline"]["cores"] >= 1 and abs(j["cpu_baseline"]["value"] - j["value"]) < 1e-9
    assert j["e2e"] == {"value": j["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert j["gpu_launches"] == 0 and "workload" in j["config"]


@pytest.mark.skipif(not _no_gpu(), reason="a CUDA device is present")
def test_product_arm_refuses_to_run_without_a_gpu():
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--steps", "1", "--warmup", "1", "--frames-per-gpu", "2", "--no-e2e", "--no-cpu-baseline"],
                         capture_output=True, text=True, timeout=600, cwd=REPO)
    assert out.returncode != 0
    assert "no CUDA device" in (out.stderr + out.stdout) and not [l for l in out.stdout.splitlines() if l.startswith("{")]


def test_front_end_stage_slots_are_merged_only_for_the_cluster_kernel():
    """The cluster front end is one launch reported in the first of the three front-end stage slots: bench.py names it k_front and
    computes no per-kernel figure for the two empty slots; the three stand-alone kernels (PWPP_FRONT=0) keep their own names."""
    sys.path.insert(0, REPO)
    import importlib
    bench = importlib.import_module("bench")
    cluster = {"k_bin_hist": 1.2, "k_bin_scan": 0.003, "k_scatter": 0.003, "k_fit_S": 0.24, "k_emit": 0.24}
    m = bench.merge_front_stages(cluster)
    assert list(m)[0] == "k_front" and abs(m["k_front"] - 1.206) < 1e-9 and "k_bin_scan" not in m and m["k_fit_S"] == 0.24
    standalone = {"k_bin_hist": 0.66, "k_bin_scan": 0.05, "k_scatter": 0.83, "k_fit_S": 0.24}
    assert bench.merge_front_stages(standalone) == standalone
    # the committed bench line of the round carries what the driver and the judge read
    line = os.path.join(REPO, "profiles", "r02", "bench_n1.json")
    if os.path.exists(line):
        j = json.load(open(line))
        for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
                    "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"):
            assert key in j, key
        r = j["roofline"]
        assert r["bound"] == "hbm" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["traffic"] is not None and "k_front" in r["per_kernel"]
        assert j["e2e"]["h2d_bytes_per_step"] > 0 and j["e2e"]["d2h_bytes_per_step"] > 0 and j["gpu_launches"] > 0


def test_dump_outputs_writes_the_same_seeded_sample(tmp_path):
    """--dump-outputs: per-frame records of every frame, and the index lists, centers and normals of a sample of frames that is
    the same from run to run, in float64 / float32 only."""
    import numpy as np
    sys.path.insert(0, REPO)
    import importlib
    bench = importlib.import_module("bench")

    class Engine:   # the getters of pwpp_b200.Engine that dump_outputs reads; frame f: f + 1 ground points, 2 non-ground, one patch
        num_ground = staticmethod(lambda f: f + 1)
        num_nonground = staticmethod(lambda f: 2)
        num_patches = staticmethod(lambda f: 1)
        height = staticmethod(lambda f: 1.5 + f)
        ground_indices = staticmethod(lambda f: np.arange(f + 1, dtype=np.int32))
        nonground_indices = staticmethod(lambda f: np.array([f + 1, f + 2], np.int32))
        centers = staticmethod(lambda f: np.full((1, 3), f, np.float32))
        normals = staticmethod(lambda f: np.full((1, 3), -f, np.float32))

    for d in ("a", "b"):
        bench.dump_outputs(Engine(), 100, str(tmp_path / d))
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) and "ground_indices.npy" in names and "num_ground.npy" in names
    out = {}
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype in (np.float32, np.float64) and a.dtype == b.dtype and np.array_equal(a, b), n
        out[n[:-4]] = a
    sample = out["sample_frames"].astype(int)
    assert len(sample) == bench.DUMP_SAMPLE_FRAMES and np.all(np.diff(sample) > 0)
    assert np.array_equal(out["num_ground"], np.arange(1, 101)) and np.array_equal(out["height"], 1.5 + np.arange(100))
    assert np.array_equal(out["ground_indices"], np.concatenate([np.arange(f + 1) for f in sample]))
    assert np.array_equal(out["nonground_indices"], np.concatenate([[f + 1, f + 2] for f in sample]))
    assert np.array_equal(out["centers"][:, 0], sample) and out["normals"].shape == (len(sample), 3)
