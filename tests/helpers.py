"""Shared comparison helpers for the parity tests."""
import ctypes as C
import hashlib
import os

import numpy as np

import oracle_py as O
from oracle_py import _Base
from pwpp_ctypes import PwppBinResult, PwppParams, default_params

HERE = os.path.dirname(os.path.abspath(__file__))


class Twin(_Base):
    """tests/host_twin.cu: the product's host+device math run sequentially on the CPU."""

    def __init__(self, params=None):
        lib = C.CDLL(os.path.join(HERE, "_build", "libpwpp_twin.so"))
        self._bind(lib, "twin_")
        lib.twin_create.argtypes = [C.POINTER(PwppParams)]; lib.twin_create.restype = C.c_void_p
        lib.twin_bin_ids.argtypes = [C.c_void_p, C.c_void_p]
        lib.twin_bin_results.argtypes = [C.c_void_p, C.c_void_p]
        lib.twin_num_bins.argtypes = [C.c_void_p]
        lib.twin_uses_fast_binning.argtypes = [C.c_void_p]
        lib.twin_fast_mismatches.argtypes = [C.c_void_p]; lib.twin_fast_mismatches.restype = C.c_longlong
        self._lib = lib
        self.params = params if params is not None else default_params()
        self._h = lib.twin_create(C.byref(self.params))
        self.nbins = lib.twin_num_bins(self._h)

    def bin_ids(self):
        out = np.empty(self._n, dtype=np.uint16)
        self._lib.twin_bin_ids(self._h, out.ctypes.data)
        return out

    def bin_results(self):
        arr = (PwppBinResult * self.nbins)()
        self._lib.twin_bin_results(self._h, C.byref(arr))
        return arr

    def fast_mismatches(self):
        return self._lib.twin_fast_mismatches(self._h)


# Everything the reference surface exposes after an estimate (including emission order), the adaptive state and its
# histories; then the label SETS (the index lists sorted).
SURFACE = ("getGroundIndices", "getNongroundIndices", "getGround", "getNonground", "getCenters", "getNormals", "state",
           "history_sizes") + tuple(f"history_{r}_{w}" for r in range(4) for w in (0, 1))
SETS = ("ground_set", "nonground_set")


def surface_array(obj, name):
    """One entry of SURFACE + SETS of an oracle / reference / twin object that has just estimated a frame."""
    if name.startswith("get"):
        return getattr(obj, name)()
    if name in SETS:
        return np.sort(obj.getGroundIndices() if name == "ground_set" else obj.getNongroundIndices())
    st = obj.state()
    if name == "state":
        return np.array([st.sensor_height, *st.elevation_thr, *st.flatness_thr], dtype=np.float64)
    if name == "history_sizes":
        return np.array([*st.n_elevation, *st.n_flatness], dtype=np.int32)
    _, r, w = name.split("_")
    return obj.history(int(r), int(w))


def digest(a) -> np.ndarray:
    """16-byte BLAKE2b of an array's dtype, shape and bytes: equal digests mean bit-identical arrays."""
    a = np.ascontiguousarray(a)
    h = hashlib.blake2b(f"{a.dtype.str}{a.shape}".encode(), digest_size=16)
    h.update(a.tobytes())
    return np.frombuffer(h.digest(), dtype=np.uint8)


class ReferenceOutputs:
    """tests/golden/reference_outputs.npz, written by tests/golden/make_golden.py: what the reference's own estimateGround
    returned on the inputs of the tests that compare with it. Per case: digests of the input and of every SURFACE + SETS
    array; for the synthetic batches also the ground mask of every frame, so that differing labels can be counted."""

    def __init__(self, path):
        z = np.load(path)
        self._digests = dict(zip(z["digest_keys"].tolist(), z["digests"]))
        self._arrays = {k: z[k] for k in z.files if k not in ("digest_keys", "digests")}

    def digest(self, case, name):
        return self._digests[f"{case}|{name}"]

    def check_input(self, case, a):
        assert np.array_equal(digest(np.ascontiguousarray(a, dtype=np.float32)), self.digest(case, "input")), \
            f"{case}: not the input the reference outputs were recorded on"

    def assert_matches(self, case, a, obj, names=SURFACE):
        """obj, which has just estimated `a`, returns bit for bit what the reference returned on this case."""
        self.check_input(case, a)
        for name in names:
            assert np.array_equal(digest(surface_array(obj, name)), self.digest(case, name)), f"{case}: {name} differs from the reference"

    def ground_masks(self, batch):
        """The reference's ground mask of every frame of a recorded batch, and the number of points it emitted per frame."""
        n = self._arrays[batch + "/n"]
        bits = np.unpackbits(self._arrays[batch + "/ground_mask"])[:n.sum()].astype(bool)
        return np.split(bits, np.cumsum(n)[:-1]), self._arrays[batch + "/emitted"]


# Inputs built by hand for the comparisons with the reference (also used by tests/golden/make_golden.py).
def edge_inputs():
    rng = np.random.default_rng(7)
    return {
        "empty": np.zeros((0, 4), np.float32),
        "one_point": np.array([[5, 0, -1.7, 0.5]], np.float32),
        "nine_in_one_bin": np.c_[5 + rng.random(9) * 0.1, rng.random(9) * 0.1, -1.7 + rng.random(9) * 0.01, rng.random(9)].astype(np.float32),
        "all_out_of_range": np.c_[rng.random((50, 2)) * 1.0, rng.random((50, 2))].astype(np.float32),
        "flat_plane": np.c_[(rng.random((5000, 2)) - 0.5) * 60, np.full(5000, -1.723), rng.random(5000)].astype(np.float32),
        "axis_points": np.array([[10, 0, -1.7, .5], [-10, 0, -1.7, .5], [0, 10, -1.7, .5], [0, -10, -1.7, .5], [3, -0.0, -1.7, .5]] * 4, np.float32),
    }


def wall_frame():
    """A wall inside a zone-0 bin: R-VPF removes points in several iterations."""
    rng = np.random.default_rng(11)
    return np.r_[np.c_[4 + rng.random(6000) * 0.05, rng.random(6000) * 0.6, -1.7 + rng.random(6000) * 2.0, rng.random(6000)],
                 np.c_[3 + rng.random(6000) * 4, rng.random(6000) * 0.6, -1.7 + rng.normal(0, 0.02, 6000), rng.random(6000)]].astype(np.float32)


def ties_frame():
    """A synthetic scan with centimetre-quantised z: thousands of exact ties per bin."""
    import synth
    b = synth.make_frame(20260922, 1).numpy()
    b[:, 2] = np.round(b[:, 2] / 0.01) * 0.01
    return b


FLAT_PATCH_SIZES = [10, 15, 16, 17, 31, 33, 63, 64, 65, 127, 129, 255, 256, 257, 511, 512, 513, 1023, 1025, 2047, 2048, 2049, 4095,
                    4096, 4097, 8191, 8192]


def flat_patch_frames():
    """One flat patch per frame, of each of FLAT_PATCH_SIZES points."""
    rng = np.random.default_rng(5)
    return [np.c_[5 + rng.random(n) * 0.5, rng.random(n) * 0.5, -1.7 + rng.normal(0, 0.03, n), rng.random(n)].astype(np.float32)
            for n in FLAT_PATCH_SIZES]


# stated floating-point tolerances of the CANON64 contract (DESIGN.md §3)
TOL_NORMAL = 1e-9       # |delta| per component of a unit normal, device/twin vs oracle (both double)
TOL_MEAN = 1e-9         # metres
TOL_SV_REL = 1e-6       # relative to the largest singular value of the patch
TOL_STATE = 1e-9        # sensor height / elevation thresholds (m); flatness thresholds relative 1e-6


def assert_sets_equal(g_a, ng_a, g_b, ng_b, n, what=""):
    """Index SETS identical and a partition of [0, n)."""
    ga, gb = np.sort(np.asarray(g_a)), np.sort(np.asarray(g_b))
    na, nbb = np.sort(np.asarray(ng_a)), np.sort(np.asarray(ng_b))
    assert ga.shape == gb.shape and np.array_equal(ga, gb), f"{what}: ground index sets differ ({len(ga)} vs {len(gb)}; sym diff {len(np.setxor1d(ga, gb))})"
    assert na.shape == nbb.shape and np.array_equal(na, nbb), f"{what}: non-ground index sets differ"
    allidx = np.concatenate([ga, na])
    assert len(np.unique(allidx)) == len(allidx), f"{what}: an index appears twice"


def assert_bins_close(ba, bb, nbins, what=""):
    for b in range(nbins):
        x, y = ba[b], bb[b]
        assert (x.n, x.n_ground, x.verdict, x.fitted) == (y.n, y.n_ground, y.verdict, y.fitted), \
            f"{what} bin {b}: (n,n_ground,verdict,fitted) {(x.n, x.n_ground, x.verdict, x.fitted)} vs {(y.n, y.n_ground, y.verdict, y.fitted)}"
        if not x.fitted or x.n == 0:
            continue
        smax = max(abs(x.sv[0]), 1e-300)
        for k in range(3):
            if np.isnan(x.sv[k]) or np.isnan(y.sv[k]):
                assert np.isnan(x.sv[k]) and np.isnan(y.sv[k]), f"{what} bin {b}: NaN singular value mismatch"
                continue
            assert abs(x.normal[k] - y.normal[k]) <= TOL_NORMAL, f"{what} bin {b} normal[{k}] {x.normal[k]} vs {y.normal[k]}"
            assert abs(x.mean[k] - y.mean[k]) <= TOL_MEAN, f"{what} bin {b} mean[{k}] {x.mean[k]} vs {y.mean[k]}"
            assert abs(x.sv[k] - y.sv[k]) <= TOL_SV_REL * smax, f"{what} bin {b} sv[{k}] {x.sv[k]} vs {y.sv[k]}"


def assert_state_close(sa, sb, what=""):
    assert abs(sa.sensor_height - sb.sensor_height) <= TOL_STATE, f"{what} sensor_height {sa.sensor_height} vs {sb.sensor_height}"
    for i in range(4):
        assert abs(sa.elevation_thr[i] - sb.elevation_thr[i]) <= TOL_STATE, f"{what} elevation_thr[{i}]"
        assert abs(sa.flatness_thr[i] - sb.flatness_thr[i]) <= 1e-6 * max(abs(sb.flatness_thr[i]), 1e-12), f"{what} flatness_thr[{i}]"
    assert list(sa.n_elevation) == list(sb.n_elevation) and list(sa.n_flatness) == list(sb.n_flatness), f"{what} history sizes"


class SimtTwin(_Base):
    """tests/simt/simt_twin.cpp: the CUDA kernels themselves, executed on the CPU by the fiber-based SIMT stand-in."""

    def __init__(self, params=None, num_streams=1, **options):
        lib = C.CDLL(os.path.join(HERE, "_build", "libpwpp_simt.so"))
        self._bind(lib, "simt_")
        lib.simt_create.argtypes = [C.POINTER(PwppParams), C.c_int]; lib.simt_create.restype = C.c_void_p
        lib.simt_bin_ids.argtypes = [C.c_void_p, C.c_void_p]
        lib.simt_bin_results.argtypes = [C.c_void_p, C.c_void_p]
        lib.simt_num_bins.argtypes = [C.c_void_p]
        lib.simt_select.argtypes = [C.c_void_p, C.c_int]
        lib.simt_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        lib.simt_queue_sizes.argtypes = [C.c_void_p]; lib.simt_queue_sizes.restype = C.c_char_p
        lib.simt_estimate_multi.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        lib.simt_set_sched_seed.argtypes = [C.c_ulonglong]
        self._lib = lib
        self.params = params if params is not None else default_params()
        self._h = lib.simt_create(C.byref(self.params), num_streams)
        self.nbins = lib.simt_num_bins(self._h)
        self._ns = [0] * num_streams
        for k, v in options.items():
            assert lib.simt_set_option(self._h, k.encode(), int(v)) == 0, k

    def estimate(self, pts):
        super().estimate(pts)
        self._ns[0] = self._n

    def estimate_multi(self, frames):
        frames = [np.ascontiguousarray(a, dtype=np.float32) for a in frames]
        cols = frames[0].shape[1]
        ptrs = (C.c_void_p * len(frames))(*[a.ctypes.data for a in frames])
        ns = (C.c_int64 * len(frames))(*[a.shape[0] for a in frames])
        self._lib.simt_estimate_multi(self._h, len(frames), ptrs, ns, cols)
        self._ns[:len(frames)] = [a.shape[0] for a in frames]
        self.select(0)

    def select(self, f):
        self._lib.simt_select(self._h, f)
        self._n = self._ns[f]

    def set_sched_seed(self, seed: int):
        """Non-zero: concurrently live CTAs are interleaved at random (per seed) instead of round-robin. Process-wide."""
        self._lib.simt_set_sched_seed(seed)

    def queue_sizes(self):
        return self._lib.simt_queue_sizes(self._h).decode()

    def bin_ids(self):
        out = np.empty(self._n, dtype=np.uint16)
        self._lib.simt_bin_ids(self._h, out.ctypes.data)
        return out

    def bin_results(self):
        arr = (PwppBinResult * self.nbins)()
        self._lib.simt_bin_results(self._h, C.byref(arr))
        return arr
