"""Generates the committed golden fixtures from a checkout of the reference project (Patchwork++).

Inputs : the reference's six KITTI scans, <checkout>/data/00000{0..5}.bin (N x 4 float32), and its
         cpp/patchworkpp/src/patchworkpp.cpp, compiled by oracle/Makefile against oracle/eigen_shim into
         oracle/_ref/libpwref.so (unmodified) and oracle/_ref/libpwref_stable.so (per-bin sort made stable so that fp32
         sums are reproducible, see oracle/ref_capi.cpp; the unmodified build is asserted to give the same label sets).
Outputs: tests/golden/kitti_00000X_{a,b}.npz  the scans themselves, column-major for better compression, split into two
                                        halves of the points so that every file stays under 1 MB
         tests/golden/golden_ref.npz    outputs of the reference's OWN estimateGround for three parameter sets x {fresh
                                        instance per scan, one instance over the six scans in order}:
                                          ground masks (bit-packed), centers, normals, adaptive state after every scan.
         tests/golden/reference_outputs.npz  what the tests that compare with the reference bit for bit need
                                        (helpers.ReferenceOutputs): digests of everything the stable-sort build returned on
                                        the fixtures, synthetic scans and hand-built inputs of test_oracle_vs_reference.py,
                                        test_order.py and test_gpu_reference.py; ground masks of the unmodified build on the
                                        synthetic batches whose differing labels test_gpu_reference.py counts.
Usage: python tests/golden/make_golden.py REFERENCE_CHECKOUT
"""
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(REPO, "oracle"))
sys.path.insert(0, os.path.join(REPO, "tests"))
import oracle_py as O  # noqa: E402
import synth  # noqa: E402  (oracle_py puts patchwork-plusplus_b200/ on the path)
from helpers import SETS, SURFACE, FLAT_PATCH_SIZES, digest, edge_inputs, flat_patch_frames, surface_array, ties_frame, wall_frame  # noqa: E402
from param_sets import PARAM_SETS  # noqa: E402

SEED = 20260922   # the synthetic scans of the benchmark and of test_gpu_reference.py


def golden_ref(scans):
    out = {}
    for pname, (mk, cols) in PARAM_SETS.items():
        for mode in ("fresh", "seq"):
            ref = O.Reference(mk(), stable_sort=True)
            raw = O.Reference(mk(), stable_sort=False)  # the unmodified reference (std::sort)
            for f, a in enumerate(scans):
                if mode == "fresh":
                    ref = O.Reference(mk(), stable_sort=True)
                    raw = O.Reference(mk(), stable_sort=False)
                ref.estimate(a[:, :cols])
                raw.estimate(a[:, :cols])
                # tie order of the per-bin sort must not change any label
                assert np.array_equal(np.sort(raw.getGroundIndices()), np.sort(ref.getGroundIndices()))
                g = ref.getGroundIndices()
                ng = ref.getNongroundIndices()
                mask = np.zeros(a.shape[0], dtype=bool)
                mask[g] = True
                assert len(g) + len(ng) == a.shape[0] and len(np.unique(np.concatenate([g, ng]))) == a.shape[0]
                st = ref.state()
                k = f"{pname}/{mode}/{f}"
                out[k + "/ground_mask"] = np.packbits(mask)
                out[k + "/n_ground"] = np.int64(len(g))
                out[k + "/centers"] = ref.getCenters()
                out[k + "/normals"] = ref.getNormals()
                out[k + "/state"] = np.array([st.sensor_height, *st.elevation_thr, *st.flatness_thr], dtype=np.float64)
                out[k + "/hist_n"] = np.array([*st.n_elevation, *st.n_flatness], dtype=np.int32)
                print(k, len(g), len(ng), ref._f("num_patches")(ref._h), st.sensor_height)
    np.savez_compressed(os.path.join(HERE, "golden_ref.npz"), **out)


def reference_outputs(scans):
    keys, digests, arrays = [], [], {}

    def record(case, a, ref, names=SURFACE + SETS):
        for name, x in [("input", np.ascontiguousarray(a, dtype=np.float32))] + [(n, surface_array(ref, n)) for n in names]:
            keys.append(f"{case}|{name}")
            digests.append(digest(x))

    def stable(a, params=None):
        ref = O.Reference(params, stable_sort=True)
        ref.estimate(a)
        return ref

    for pname, (mk, cols) in PARAM_SETS.items():
        for mode in ("fresh", "seq"):
            ref = O.Reference(mk(), stable_sort=True)
            for f, a in enumerate(scans):
                if mode == "fresh":
                    ref = O.Reference(mk(), stable_sort=True)
                ref.estimate(a[:, :cols])
                record(f"kitti{f}/{pname}/{mode}", a[:, :cols], ref)
    raw = O.Reference(stable_sort=False)
    raw.estimate(scans[0])
    record("kitti0/default/std_sort", scans[0], raw, SETS)
    ref = O.Reference(stable_sort=True)
    for f in range(4):
        a = synth.make_frame(1234, f).numpy()
        ref.estimate(a)
        record(f"synth1234_{f}/seq", a, ref)
    for name, a in edge_inputs().items():
        record(f"edge/{name}", a, stable(a))
    record("wall", wall_frame(), stable(wall_frame()))
    record("ties", ties_frame(), stable(ties_frame()))
    for n, a in zip(FLAT_PATCH_SIZES, flat_patch_frames()):
        record(f"flat{n}", a, stable(a))
    for f in range(6):
        a = synth.make_frame(SEED, f).numpy()
        record(f"synth{f}", a, stable(a))
    a = synth.make_frame(SEED, 1, "dense1m").numpy()
    record("dense1", a, stable(a))

    # label masks of the unmodified reference on the synthetic batches
    for batch, frames in (("config3", [(f, "kitti64") for f in range(256)]), ("dense", [(0, "dense1m")])):
        masks, ns, emitted = [], [], []
        for f, sensor in frames:
            a = synth.make_frame(SEED, f, sensor).numpy()
            raw = O.Reference(stable_sort=False)
            raw.estimate(a)
            m = np.zeros(len(a), bool)
            m[raw.getGroundIndices()] = True
            masks.append(m)
            ns.append(len(a))
            emitted.append(len(raw.getGroundIndices()) + len(raw.getNongroundIndices()))
            record(f"{batch}/{f}", a, raw, ())
            raw.close()
        arrays[batch + "/ground_mask"] = np.packbits(np.concatenate(masks))
        arrays[batch + "/n"] = np.array(ns, np.int64)
        arrays[batch + "/emitted"] = np.array(emitted, np.int64)
    np.savez_compressed(os.path.join(HERE, "reference_outputs.npz"), digest_keys=np.array(keys), digests=np.array(digests), **arrays)


def main(checkout):
    O.build()
    subprocess.check_call(["make", "-C", os.path.join(REPO, "oracle"), "ref", "REFERENCE=" + os.path.abspath(checkout)], stdout=subprocess.DEVNULL)
    scans = []
    for f in range(6):
        a = np.fromfile(os.path.join(checkout, "data", f"{f:06d}.bin"), dtype=np.float32).reshape(-1, 4)
        scans.append(a)
        half = (len(a) + 1) // 2
        for h, part in zip("ab", (a[:half], a[half:])):
            np.savez_compressed(os.path.join(HERE, f"kitti_{f:06d}_{h}.npz"), xyzi_t=np.ascontiguousarray(part.T))
    golden_ref(scans)
    reference_outputs(scans)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
