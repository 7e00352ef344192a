"""CPU: pins the trajectory replay of tests/evaluate_model.py (replay_track) on the oracle's own runs.

A traced run records, per iteration, the level, J^T r, delta_p, normdp and the visible points.  The pose of every
measurement is p_in's internal fp32 coefficients plus the running fp32 sum of the recorded steps, so the CPU model can
measure again at exactly that pose.  On the oracle's trajectories, in sum modes 0 and 1, every record must come out bit
for bit, and so must the final pose through getPose_se3 (donorm included); the records must satisfy the exact
structure checks (helpers.check_trajectory) that tests/test_gpu_replay.py applies to every kernel.
"""
import numpy as np
import pytest

from helpers import make_case, oracle_run, replay_models, check_trajectory, replay_trace_cap
from evaluate_model import replay_batch

P_SHIFT = [1.2, 0.3, 0.0, 0.0, 0.02, 0.0]          # pushes border points out of the new frame mid-level

# (id, case options, p_in of every track)
CASES = [
    ("donorm", dict(seed=301, psz=8, npts=30, lv_f=2, donorm=1, ntracks=2), [0.01, -0.02, 0.005, 0.002, -0.001, 0.003]),
    ("donorm-patchnorm", dict(seed=302, psz=8, npts=24, lv_f=2, donorm=1, dopatchnorm=1), None),
    ("psz4-cap", dict(seed=303, psz=4, npts=50, lv_f=2, maxpttrack=32), None),
    ("psz7-patchnorm", dict(seed=304, psz=7, npts=20, lv_f=2, dopatchnorm=1), None),
    ("psz16-lvl1", dict(seed=305, psz=16, npts=10, lv_f=3, lv_l=1, w=960, h=544), None),
    ("psz32", dict(seed=306, psz=32, npts=5, lv_f=2, w=1280, h=704), None),
    ("large-motion", dict(seed=307, psz=8, npts=40, lv_f=2, scale=4.0), P_SHIFT),
    ("dense-psz1", dict(seed=308, w=160, h=120, lv_f=1, psz=1, dense_border=40, tilt=(0.1, -0.08)), None),
]


def replay_oracle(orc, c, p_in, mode):
    """The oracle's traced run in sum mode `mode` and the model's replay of it in the same mode."""
    cap = replay_trace_cap(c["op"])
    o = oracle_run(orc, c, trace_cap=cap, sum_mode=mode, p_in=p_in)
    models = replay_models(orc, c, o["pyr"], p_in)
    orc.set_sum_mode(mode)
    try:
        rep = replay_batch(models, o["trace"])
    finally:
        orc.set_sum_mode(0)
    return o, rep


def assert_replay_exact(o, rep, op):
    check_trajectory(o, op)
    tr = o["trace"]
    for t in range(tr.shape[0]):
        for k in range(int((tr[t, :, 0] >= 0).sum())):
            assert np.array_equal(rep["trace"][t, k, :16], tr[t, k, :16]), (t, k, rep["trace"][t, k], tr[t, k])
            # jabs: the same fp64 terms, summed per point there and in one pass here
            assert np.allclose(rep["trace"][t, k, 16:22], tr[t, k, 16:22], rtol=1e-6, atol=0), (t, k)
    assert np.array_equal(rep["p_out"], o["p_out"]), (rep["p_out"], o["p_out"])


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("k", range(len(CASES)), ids=[c[0] for c in CASES])
def test_replay_bit_identical(orc, k, mode):
    _, kw, p = CASES[k]
    c = make_case(**kw)
    p_in = None if p is None else np.tile(np.asarray(p, np.float64), (c["T"], 1))
    o, rep = replay_oracle(orc, c, p_in, mode)
    assert_replay_exact(o, rep, c["op"])


@pytest.mark.parametrize("mode", [0, 1])
def test_replay_uneven_batch(orc, mode):
    """Tracks of 0, 1, 17 and 40 points, the last one above the maxpttrack cap and shifted out of the frame."""
    c = make_case(seed=309, psz=8, npts=40, lv_f=2, maxpttrack=32)
    sizes = [0, 1, 17, 40]
    c["pts"] = np.concatenate([c["sc"].points(700 + t, n, 8, 2) for t, n in enumerate(sizes)])
    c["pt_off"] = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    c["T"] = len(sizes)
    p_in = np.zeros((4, 6))
    p_in[3] = P_SHIFT
    o, rep = replay_oracle(orc, c, p_in, mode)
    assert_replay_exact(o, rep, c["op"])
    assert (o["trace"][0, :, 2:14] == 0).all() and o["npixres"][0] == 0


def test_replay_detects_a_wrong_step(orc):
    """The replay measures at the recorded trajectory: a step changed by 1e-3 moves every later measurement."""
    _, kw, p = CASES[6]
    c = make_case(**kw)
    o, _ = replay_oracle(orc, c, None, 0)
    bad = o["trace"].copy()
    bad[0, 0, 8] *= np.float32(1.001)
    rep = replay_batch(replay_models(orc, c, o["pyr"]), bad)
    n = int((bad[0, :, 0] >= 0).sum())
    assert np.array_equal(rep["trace"][0, 0, :16], o["trace"][0, 0, :16])
    assert all(not np.array_equal(rep["trace"][0, k, 2:8], o["trace"][0, k, 2:8]) for k in range(1, n))
