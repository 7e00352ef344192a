"""CPU: the oracle restatement against stored outputs on the seeded cases on which it was compared with the
reference's OWN sources (oracle/_ref: the reference compiled against the stand-in headers), bit-exact throughout.

tests/golden/vs_ref.npz holds the ORACLE's outputs on these cases, not the reference's: the reference's sources are
not part of this repository and were not at hand when the file was recorded, so it pins the oracle against change
here, while tests/test_oracle_golden.py pins it against outputs the reference itself produced.  Wherever oracle/_ref
is built (`make -C oracle ref REF=<reference checkout>`), the reference's outputs are checked against the same stored
values, which is the original comparison and also verifies the file.

The inputs are regenerated from their seeds by invcompcamtrack_b200.synth, whose blur uses scipy.ndimage (its numpy
fallback gives other images), so scipy is needed; digests of the inputs are stored beside the outputs so that other
inputs are reported as such and not as a change of the oracle."""
import os

import numpy as np
import pytest

from oracle import oracle as O
from helpers import REF_CAMERAS, REF_CASES, ref_outputs

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "vs_ref.npz")


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


@pytest.fixture(scope="module")
def computed(orc):
    """The oracle's outputs, and the reference's where oracle/_ref is built."""
    libs = {"oracle": orc}
    if O.RefLib.available():
        libs["reference"] = O.RefLib()
    return {name: ref_outputs(lib, orc) for name, lib in libs.items()}


@pytest.mark.parametrize("kw", REF_CASES)
def test_trace_bit_identical(computed, gold, kw):
    k = REF_CASES.index(kw)
    for lib, got in computed.items():
        assert got["t%d_inputs" % k] == str(gold["t%d_inputs" % k]), \
            "the seeded inputs changed (invcompcamtrack_b200.synth; is scipy installed?)"
        assert np.array_equal(got["t%d_pyr_sample" % k], gold["t%d_pyr_sample" % k]), lib
        assert got["t%d_pyr" % k] == str(gold["t%d_pyr" % k]), lib
        for name in ("p", "jtr", "dp", "q", "pts"):
            assert np.array_equal(got["t%d_%s" % (k, name)], gold["t%d_%s" % (k, name)], equal_nan=True), (lib, name)


def test_camera_levels(computed, gold):
    for lib, got in computed.items():
        for k in range(len(REF_CAMERAS)):
            assert np.array_equal(got["camera%d" % k], gold["camera%d" % k]), lib


def test_batch_poses_identical(computed, gold):
    for lib, got in computed.items():
        assert np.array_equal(got["batch_p_out"], gold["batch_p_out"]), lib
