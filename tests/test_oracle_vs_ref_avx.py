"""CPU: the oracle's sum mode 1 — Eigen's vectorised .sum() on 8-float AVX packets, sixteen chains — against stored
outputs on the seeded cases of tests/test_oracle_vs_ref.py (helpers.REF_CASES, the camera levels and the 12-track
batch), bit-exact throughout.  Sum order 3 of the library (ict_tracker_set_sum_order) reproduces this mode.

tests/golden/vs_ref_avx.npz holds the ORACLE's outputs in sum mode 1, not the reference's, with the same caveat as
vs_ref.npz: the reference's sources are not part of this repository, so without them the file pins the oracle's
mode 1 against change.  Wherever oracle/_ref_avx is built (`make -C oracle -f shim_avx/ref_avx.mk
REF=<reference checkout>`: the reference's unmodified sources against the stand-in Eigen with its dynamic-size sums
on 8-float packets, oracle/shim_avx/packet8_sum.h), the reference's outputs are checked against the same stored
values.

    python tests/test_oracle_vs_ref_avx.py      # re-records the file from the oracle in sum mode 1
"""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
if __name__ == "__main__":
    sys.path[:0] = [HERE, os.path.dirname(HERE)]

from oracle import oracle as O
from helpers import REF_CAMERAS, REF_CASES, ref_outputs

GOLD = os.path.join(HERE, "golden", "vs_ref_avx.npz")
REF_AVX = os.path.join(os.path.dirname(O.__file__), "_ref_avx", "libictrack_ref.so")


def oracle_avx_outputs(orc):
    orc.set_sum_mode(1)
    try:
        return ref_outputs(orc, orc)
    finally:
        orc.set_sum_mode(0)


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


@pytest.fixture(scope="module")
def computed(orc):
    """The oracle's outputs in sum mode 1, and the AVX-packet reference's where oracle/_ref_avx is built."""
    out = {"oracle": oracle_avx_outputs(orc)}
    if os.path.exists(REF_AVX):
        out["reference_avx"] = ref_outputs(O.RefLib(REF_AVX), orc)
    return out


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


def test_packet_orders_differ(computed):
    """The stored cases tell the two packet widths apart: mode 1 is not mode 0 on them."""
    sse = np.load(os.path.join(HERE, "golden", "vs_ref.npz"))
    got = computed["oracle"]
    assert any(not np.array_equal(got["t%d_jtr" % k], sse["t%d_jtr" % k]) for k in range(len(REF_CASES)))


SUM_PROBE = r"""
#include <Eigen/Dense>
#include <cmath>
#include <cstdio>
#include <cstdlib>
int main(int argc, char** argv) {
  const int n = argc - 1;
  float* v = (float*)malloc(sizeof(float) * (n + 1));
  for (int i = 0; i < n; ++i) v[i] = (float)strtod(argv[i + 1], 0);
  Eigen::Map<Eigen::MatrixXf> m(v, n, 1);
  const float s = m.sum(), q = m.norm();
  printf("%a %a\n", s, q);
  return 0;
}
"""


@pytest.mark.parametrize("n", [0, 5, 8, 12, 16, 24, 40, 64, 100, 333])
def test_stand_in_packet_sums_equal_the_oracle(orc, tmp_path, n):
    """The stand-in Eigen (oracle/shim) sums on 4-float packets like the oracle's mode 0; with
    oracle/shim_avx/packet8_sum.h forced in (the oracle/_ref_avx build) it sums on 8-float packets like mode 1 —
    .sum() and .norm() of a dynamic-size float vector, bit for bit."""
    import shutil
    import subprocess
    if shutil.which("g++") is None:
        pytest.skip("no C++ compiler")
    odir = os.path.dirname(O.__file__)
    src = tmp_path / "probe.cpp"
    src.write_text(SUM_PROBE)
    v = (np.random.default_rng(n).standard_normal(n) * np.logspace(0, 3, n)).astype(np.float32)
    args = ["%.9g" % x for x in v]
    for mode, extra in ((0, []), (1, ["-include", os.path.join(odir, "shim_avx", "packet8_sum.h")])):
        exe = tmp_path / ("probe%d" % mode)
        subprocess.run(["g++", "-O3", "-msse4", "-mavx", "-ffp-contract=off", "-std=c++11", "-w"] + extra +
                       ["-I", os.path.join(odir, "shim"), str(src), "-o", str(exe)], check=True)
        s, q = (float.fromhex(t) for t in subprocess.run([str(exe)] + args, capture_output=True, text=True,
                                                          check=True).stdout.split())
        orc.set_sum_mode(mode)
        try:
            want_s = np.float32(orc.esum(v))
            want_q = np.float32(np.sqrt(np.float32(orc.esum(v * v))))
        finally:
            orc.set_sum_mode(0)
        assert np.float32(s) == want_s and np.float32(q) == want_q, (mode, n)


if __name__ == "__main__":
    np.savez_compressed(GOLD, **oracle_avx_outputs(O.OracleLib()))
    print(GOLD)
