"""Pins the restated oracle (oracle/pwpp_oracle.c, arith=REF32) against the reference's OWN estimateGround:
reference cpp/patchworkpp/src/patchworkpp.cpp compiled unmodified against oracle/eigen_shim
(oracle/_ref/libpwref_stable.so, only the per-bin sort made stable — see oracle/ref_capi.cpp), whose outputs
tests/golden/make_golden.py recorded in tests/golden/reference_outputs.npz.
Everything must agree BIT FOR BIT, including the emission order of the index lists."""
import pytest

import oracle_py as O
from helpers import SETS, edge_inputs
from param_sets import PARAM_SETS


@pytest.mark.parametrize("pname", list(PARAM_SETS))
@pytest.mark.parametrize("mode", ["fresh", "seq"])
def test_fixtures_bit_identical(kitti, refout, pname, mode):
    mk, cols = PARAM_SETS[pname]
    orc = O.Oracle(mk(), O.ARITH_REF32)
    for f, a in enumerate(kitti):
        if mode == "fresh":
            orc = O.Oracle(mk(), O.ARITH_REF32)
        orc.estimate(a[:, :cols])
        refout.assert_matches(f"kitti{f}/{pname}/{mode}", a[:, :cols], orc)


def test_synthetic_sequence_bit_identical(refout):
    import synth
    orc = O.Oracle(arith=O.ARITH_REF32)
    for f in range(4):
        a = synth.make_frame(1234, f).numpy()
        orc.estimate(a)
        refout.assert_matches(f"synth1234_{f}/seq", a, orc)


def test_unstable_sort_only_changes_order(kitti, refout):
    """The unmodified reference (std::sort) gives the same index SETS as the stable-sort variant the oracle reproduces."""
    a = kitti[0]
    orc = O.Oracle(arith=O.ARITH_REF32)
    orc.estimate(a)
    refout.assert_matches("kitti0/default/std_sort", a, orc, SETS)


def test_edge_inputs_bit_identical(refout):
    for name, a in edge_inputs().items():
        orc = O.Oracle(arith=O.ARITH_REF32)
        orc.estimate(a)
        refout.assert_matches(f"edge/{name}", a, orc)
