import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
for p in (os.path.join(REPO, "patchwork-plusplus_b200"), os.path.join(REPO, "oracle"), HERE, os.path.join(REPO, "patchwork-plusplus_b200", "lib")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _cuda_available():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _cuda_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session", autouse=True)
def _build_checkers():
    import oracle_py
    oracle_py.build()
    build_twin()
    build_simt()


def build_twin(force=False):
    """CPU twin of the CUDA pipeline (tests/host_twin.cu), nvcc host pass; prebuilt .so travels to the GPU box."""
    out = os.path.join(HERE, "_build", "libpwpp_twin.so")
    src = os.path.join(HERE, "host_twin.cu")
    deps = [src] + [os.path.join(REPO, "patchwork-plusplus_b200", "csrc", f) for f in ("pwpp_math.cuh", "pwpp_gle.cuh", "pwpp_host.hpp")] + [os.path.join(HERE, "gle_sequential.cuh")]
    if force or not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        subprocess.check_call(["/usr/local/cuda/bin/nvcc", "-O2", "-std=c++17", "-x", "cu", "-Wno-deprecated-gpu-targets",
                               "-Xcompiler", "-fPIC,-ffp-contract=off", "-shared", "-I" + os.path.join(REPO, "include"),
                               "-I" + os.path.join(REPO, "patchwork-plusplus_b200", "csrc"), "-o", out, src])
    return out


def build_simt(force=False):
    """The CUDA kernels compiled by g++ against the SIMT stand-in (tests/simt/cuda_runtime.h) for CPU execution."""
    out = os.path.join(HERE, "_build", "libpwpp_simt.so")
    csrc = os.path.join(REPO, "patchwork-plusplus_b200", "csrc")
    deps = [os.path.join(HERE, "simt", f) for f in ("simt_twin.cpp", "cuda_runtime.h")] + \
           [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".cuh", ".hpp"))]
    if force or not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-I" + os.path.join(HERE, "simt"),
                               "-I" + os.path.join(REPO, "include"), "-I" + csrc, "-o", out, os.path.join(HERE, "simt", "simt_twin.cpp")])
    return out


def load_kitti(f: int) -> np.ndarray:
    """The reference's fixture scan data/00000f.bin (N x 4 float32), from the committed copy (two halves of the points)."""
    halves = [np.load(os.path.join(HERE, "golden", f"kitti_{f:06d}_{h}.npz"))["xyzi_t"] for h in "ab"]
    return np.ascontiguousarray(np.concatenate(halves, axis=1).T)


@pytest.fixture(scope="session")
def kitti():
    return [load_kitti(f) for f in range(6)]


@pytest.fixture(scope="session")
def golden():
    return np.load(os.path.join(HERE, "golden", "golden_ref.npz"))


@pytest.fixture(scope="session")
def refout():
    from helpers import ReferenceOutputs
    return ReferenceOutputs(os.path.join(HERE, "golden", "reference_outputs.npz"))
