"""Reference emission order (pwpp_set_output_order(PWPP_ORDER_REFERENCE), csrc/pwpp_order.cuh): the index LISTS — not just the
sets — equal those of the reference's own code with a stable per-bin sort (oracle/_ref/libpwref_stable.so: ties in z keep
ascending point index; with std::sort their order is unspecified in the reference itself), as recorded in
tests/golden/reference_outputs.npz. Kernels on the SIMT twin here, on the GPU in tests/test_gpu_reference.py."""
import numpy as np
import pytest

from helpers import FLAT_PATCH_SIZES, SimtTwin, digest, flat_patch_frames, ties_frame, wall_frame
from param_sets import PARAM_SETS

LISTS = ("getGroundIndices", "getNongroundIndices")


@pytest.mark.parametrize("patch", [0, 1])
def test_fixture_lists_in_reference_order(kitti, refout, patch):
    for f in (0, 3):
        tw = SimtTwin(order=1, patch=patch)
        tw.estimate(kitti[f])
        refout.assert_matches(f"kitti{f}/default/fresh", kitti[f], tw, LISTS)


def test_rvpf_removals_come_first_in_iteration_order(refout):
    """A wall inside a zone-0 bin: R-VPF removes points in several iterations; the reference appends them to the non-ground
    list iteration by iteration, each in ascending z, before the final rejects (patchworkpp.cpp:495-504, :529-541)."""
    wall = wall_frame()
    for patch in (0, 1):
        tw = SimtTwin(order=1, patch=patch)
        tw.estimate(wall)
        refout.assert_matches("wall", wall, tw, LISTS)


def test_other_parameter_set_and_synthetic_and_ties(refout):
    mk, cols = PARAM_SETS["no_rvpf_tgr"]
    a = np.ascontiguousarray(conftest_kitti(1)[:, :cols])
    tw = SimtTwin(mk(), order=1)
    tw.estimate(a)
    refout.assert_matches("kitti1/no_rvpf_tgr/fresh", a, tw, LISTS)
    b = ties_frame()
    tw = SimtTwin(order=1)
    tw.estimate(b)
    if np.array_equal(digest(np.sort(tw.getGroundIndices())), refout.digest("ties", "ground_set")):   # (lattice data can flip labels between fp32 and double, DESIGN.md section 3)
        refout.assert_matches("ties", b, tw, LISTS)


def conftest_kitti(f):
    import conftest
    return conftest.load_kitti(f)


def test_sort_kernels_at_their_size_limits(refout):
    """Patches whose sizes sit on the limits of the sort kernels (k_order_warp: 16-key lanes, 512-key warps; k_order_cta<128/256/512>:
    2048 / 4096 / 8192 keys) and of their padding (powers of two +- 1): one flat patch per frame, all frames in one batched call."""
    frames = flat_patch_frames()
    tw = SimtTwin(num_streams=len(frames), order=1)
    tw.estimate_multi(frames)
    for f, (n, a) in enumerate(zip(FLAT_PATCH_SIZES, frames)):
        tw.select(f)
        refout.assert_matches(f"flat{n}", a, tw, LISTS)
