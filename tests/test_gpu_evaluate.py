"""ict_track_evaluate on the GPU: one Gauss-Newton measurement per track at a chosen pose.

  * orders 1 and 3 bit-identical to the CPU model (tests/evaluate_model.py, oracle sum modes 0 and 1) in every output,
    on mixed batches (0- and 1-point tracks, per-track frame pairs of a five-frame store, poses that move points out of
    the frame), psz 1 (dense), 4, 7, 8, 16 and 32, dopatchnorm and donorm, at every level;
  * orders 0 and 2: exact visible-point counts, H / J^T r / SSR within 1e-5 of the oracle relative to the fp64 sums of
    absolute terms, the same bits on a repeated call and for each track under a permutation of the tracks;
  * after a traced ict_track_batch on every kernel family, evaluate(p_in, p_in, lv_f) is the trace's first record;
  * no side effects on later tracking calls, the 2-D points or the carried keep_state arrays; the documented errors;
  * on synthetic pairs with known motion, the residual separates tracked poses from the initial ones and from frames
    of another scene.
"""
import numpy as np
import pytest

from invcompcamtrack_b200 import synth
from oracle import oracle as O
from evaluate_model import evaluate_batch
from test_gpu_mixed_batches import (MIXED, G8, G16, G32, NFR, TC, store, make_mixed, permuted, oracle_mixed,
                                    new_tracker, gpu_mixed)

pytestmark = pytest.mark.gpu

FAST, SSE, GENERAL, AVX = 0, 1, 2, 3
OUT = ("H", "jtr", "dp", "ssr", "nvis", "pt_ssr")


def p_cur_of(c, seed):
    """A measurement pose near each track's p_in."""
    rng = np.random.default_rng(seed)
    return c["p_in"] + np.concatenate([rng.uniform(-0.004, 0.004, (c["T"], 3)), rng.uniform(-0.001, 0.001, (c["T"], 3))], 1)


def oracle_eval(orc, c, level, p_cur, mode):
    st = c["st"]
    op = O.OptParam.from_buffer_copy(bytes(c["op"]))
    orc.set_sum_mode(mode)
    try:
        return evaluate_batch(orc, op, st["sc"].fc, st["sc"].cc, st["sc"].wh, [q[0] for q in st["pyr"]],
                              [q[1] for q in st["pyr"]], [q[2] for q in st["pyr"]], c["pt_off"], c["pts"], c["rf"],
                              c["nf"], c["p_in"], p_cur, level)
    finally:
        orc.set_sum_mode(0)


def gpu_eval(ict, c, order, level, p_cur=None, fr=None):
    tr = new_tracker(ict, c, order)
    try:
        return tr.evaluate(fr or c["st"]["fr"], c["rf"], c["nf"], c["p_in"], p_cur, level, per_point=True)
    finally:
        tr.close()


def assert_equal_outputs(g, o, what=""):
    for k in OUT:
        assert np.array_equal(g[k], o[k], equal_nan=True), (what, k)


def assert_close_tree(g, o, what=""):
    """Tree order against the oracle: nvis exact, every sum within 1e-5 of its fp64 sum of absolute terms."""
    assert np.array_equal(g["nvis"], o["nvis"]), what
    iu = np.triu_indices(6)
    dH = np.abs(g["H"][:, iu[0], iu[1]].astype(np.float64) - o["H"][:, iu[0], iu[1]])
    assert (dH <= 1e-5 * o["habs"] + 1e-30).all(), (what, (dH / np.maximum(o["habs"], 1e-30)).max())
    dj = np.abs(g["jtr"].astype(np.float64) - o["jtr"])
    assert (dj <= 1e-5 * o["jabs"] + 1e-30).all(), (what, (dj / np.maximum(o["jabs"], 1e-30)).max())
    ds = np.abs(g["ssr"].astype(np.float64) - o["ssr"])
    assert (ds <= 1e-5 * o["ssr_d"] + 1e-30).all(), what
    m = o["pt_ssr"] >= 0
    assert np.array_equal(g["pt_ssr"] >= 0, m), what
    assert (np.abs(g["pt_ssr"][m].astype(np.float64) - o["pt_ssr"][m]) <= 1e-6 * o["pt_ssr"][m] + 1e-30).all(), what


# geometry, sizes, builder options: every psz the issue lists, the option combinations, uneven tracks
EVAL_CASES = [
    pytest.param(G8, [0, 1, 3, 13, 64, 100], {}, id="psz8"),
    pytest.param(G8, [1, 7, 129, 40, 0], dict(dopatchnorm=1), id="psz8-patchnorm"),
    pytest.param(G8, [1, 7, 50, 19, 1], dict(donorm=1, dopatchnorm=1), id="psz8-donorm-patchnorm"),
    pytest.param(G8, [5, 90, 17, 41, 0], dict(maxpttrack=40), id="psz8-cap40"),
    pytest.param(G16, [0, 1, 9, 17, 40], dict(donorm=1), id="psz16-donorm"),
    pytest.param(G32, [0, 1, 2, 4, 9, 13], {}, id="psz32"),
    pytest.param((4, 640, 480, 3), [0, 1, 5, 50], {}, id="psz4"),
    pytest.param((7, 640, 480, 3), [0, 1, 5, 50], dict(dopatchnorm=1), id="psz7-patchnorm"),
    pytest.param((1, 320, 240, 2), [8, 0, 1], dict(dense=0), id="dense"),
]


@pytest.mark.parametrize("geom,sizes,kw", EVAL_CASES)
def test_evaluate_against_oracle(ict, orc, geom, sizes, kw):
    st = store(ict, orc, *geom)
    c = make_mixed(ict, st, sizes, seed=300 + sum(sizes) % 97, **kw)
    perm = np.roll(np.arange(c["T"]), 1)
    cp = permuted(c, perm)
    for level in range(c["op"].lv_l, c["op"].lv_f + 1):
        p_cur = p_cur_of(c, level)
        cp_cur = p_cur[perm]
        o0, o1 = oracle_eval(orc, c, level, p_cur, 0), oracle_eval(orc, c, level, p_cur, 1)
        for order in (SSE, AVX):
            assert_equal_outputs(gpu_eval(ict, c, order, level, p_cur), o0 if order == SSE else o1, (level, order))
        for order in (FAST, GENERAL):
            g = gpu_eval(ict, c, order, level, p_cur)
            assert_close_tree(g, o0, (level, order))
            assert_equal_outputs(gpu_eval(ict, c, order, level, p_cur), g, (level, order, "repeat"))
            gp = gpu_eval(ict, cp, order, level, cp_cur)
            for k in ("H", "jtr", "dp", "ssr", "nvis"):
                assert np.array_equal(gp[k], g[k][perm], equal_nan=True), (level, order, k)
            for j, t in enumerate(perm):
                a = g["pt_ssr"][c["pt_off"][t]:c["pt_off"][t + 1]]
                assert np.array_equal(gp["pt_ssr"][cp["pt_off"][j]:cp["pt_off"][j + 1]], a), (level, order, j)
    # p_cur omitted == p_ref
    assert_equal_outputs(gpu_eval(ict, c, SSE, c["op"].lv_f), gpu_eval(ict, c, SSE, c["op"].lv_f, c["p_in"]))


def test_points_out_of_view_are_measured(ict, orc):
    """The mixed builder's pans move part or all of a track's points out of the new frame: those are counted out."""
    st = store(ict, orc, *G8)
    c = make_mixed(ict, st, [30, 30, 30, 30, 30], seed=9)
    p_cur = c["p_in"].copy()
    p_cur[3, 0] += 2.0                   # a pan of about a third of the frame at depth 5 ...
    p_cur[4, 0] += 8.0                   # ... and one past its width
    g = gpu_eval(ict, c, SSE, 0, p_cur)
    assert 0 < g["nvis"][3] < 30 and g["nvis"][4] == 0
    assert ((g["pt_ssr"] == -1).sum()) == (150 - g["nvis"].sum())


# ---- after a traced track_batch on every kernel family -------------------------------------------------------------
@pytest.mark.parametrize("geom,sizes,kw,want", MIXED)
def test_first_trace_record(ict, orc, geom, sizes, kw, want):
    st = store(ict, orc, *geom)
    c = make_mixed(ict, st, sizes, seed=sum(sizes) % 1000 + len(sizes), **kw)
    o0 = oracle_mixed(orc, c, 0)
    lv_f = c["op"].lv_f
    knob_runs = [(SSE, ()), (AVX, ()), (FAST, ()), (GENERAL, ())]
    if geom[0] == 32 and want[SSE].startswith("k_track_r"):
        knob_runs.append((SSE, (("no_k2r", 1),)))
    for order, knobs in knob_runs:
        tr = new_tracker(ict, c, order, knobs)
        try:
            r = tr.track_batch(st["fr"], c["rf"], c["nf"], c["p_in"], trace_cap=TC)
            e = tr.evaluate(st["fr"], c["rf"], c["nf"], c["p_in"], None, lv_f)
        finally:
            tr.close()
        rec = r["trace"][:, 0]
        assert np.array_equal(e["nvis"], rec[:, 15]), order
        if order in (SSE, AVX):
            assert np.array_equal(e["jtr"], rec[:, 2:8], equal_nan=True), (order, knobs)
            assert np.array_equal(e["dp"], rec[:, 8:14], equal_nan=True), (order, knobs)
            continue
        for t in range(c["T"]):     # the first-iteration gate of the tree-order kernels (tests/helpers.py check_parity)
            if np.isnan(o0["p_out"][t]).any() or c["rf"][t] == c["nf"][t] or o0["trace"][t, 0, 15] == 0:
                continue
            scale = np.maximum(o0["trace"][t, 0, 16:22].astype(np.float64), 1e-30)
            d = np.abs(e["jtr"][t].astype(np.float64) - rec[t, 2:8]) / scale
            assert d.max() <= 1e-5, (order, t, d)


# ---- no side effects -------------------------------------------------------------------------------------------------
def test_no_side_effects(ict, orc):
    st = store(ict, orc, *G8)
    c = make_mixed(ict, st, [0, 1, 13, 64, 100], seed=31)
    for order in (SSE, FAST):
        ref = gpu_mixed(ict, c, order)
        tr = new_tracker(ict, c, order)
        tr.evaluate(st["fr"], c["rf"], c["nf"], c["p_in"] * 0.5, c["p_in"], 1, per_point=True)
        out = tr.track_batch(st["fr"], c["rf"], c["nf"], c["p_in"], trace_cap=TC)
        out["pt2d"] = tr.get_2dpoints()
        tr.evaluate(st["fr"], c["nf"], c["rf"], c["p_in"], None, 0)
        assert np.array_equal(tr.get_2dpoints(), out["pt2d"])       # get_2dpoints: the last SetPose's, not evaluate's
        tr.close()
        for k in ("p_out", "iters", "npixres", "pt2d"):
            assert np.array_equal(out[k], ref[k], equal_nan=True), (order, k)
        assert np.array_equal(out["trace"][..., :16], ref["trace"][..., :16], equal_nan=True)
    # keep_state: a chain of three steps with an evaluate between every two gives the bits of one without
    runs = []
    for with_eval in (False, True):
        tr = new_tracker(ict, c, SSE, knobs=(("keep_state", 1),))
        p = c["p_in"]
        poses = []
        for k in range(3):
            if with_eval:
                tr.evaluate(st["fr"], np.full(c["T"], k + 1), np.full(c["T"], k), p, None, 2)
            p = tr.track_batch(st["fr"], np.full(c["T"], k), np.full(c["T"], k + 1), p)["p_out"]
            poses.append(p)
        tr.close()
        runs.append(np.stack(poses))
    assert np.array_equal(runs[0], runs[1], equal_nan=True)


def test_errors(ict, orc):
    st = store(ict, orc, *G8)
    c = make_mixed(ict, st, [5, 9], seed=41)
    tr = new_tracker(ict, c, SSE)
    ev = lambda **kw: tr.evaluate(st["fr"], kw.get("rf", c["rf"]), c["nf"], c["p_in"], None, kw.get("level"))  # noqa
    for bad in (dict(level=c["op"].lv_f + 1), dict(level=c["op"].lv_l - 1), dict(rf=np.array([0, NFR]))):
        with pytest.raises(ict.IctError, match="ICT_ERR_BAD_ARG"):
            ev(**bad)
    tr.set_robust(ict.api.ROBUST_FULL_STEP)
    with pytest.raises(ict.IctError, match="ICT_ERR_UNSUPPORTED"):
        ev()
    tr.set_robust(0)
    ev()
    op = ict.OptParam.from_buffer_copy(bytes(c["op"]))
    op.maxpttrack = 4
    tr.set_optparam(op)
    with pytest.raises(ict.IctError, match="ICT_ERR_BAD_ARG"):
        ev()
    tr.close()


def test_points_from_device_memory(ict, orc):
    torch = pytest.importorskip("torch")
    st = store(ict, orc, *G8)
    c = make_mixed(ict, st, [0, 3, 20, 7], seed=51)
    a = gpu_eval(ict, c, SSE, 1, p_cur_of(c, 1))
    tr = ict.Tracker(ict.OptParam.from_buffer_copy(bytes(c["op"])), st["sc"].fc, st["sc"].cc, st["sc"].wh)
    off = torch.from_numpy(c["pt_off"]).cuda()
    pts = torch.from_numpy(c["pts"]).cuda()
    torch.cuda.synchronize()
    tr.set_points_dev(c["T"], off.data_ptr(), pts.data_ptr(), int(c["pt_off"][-1]), max(c["sizes"]))
    b = tr.evaluate(st["fr"], c["rf"], c["nf"], c["p_in"], p_cur_of(c, 1), 1, per_point=True)
    tr.close()
    assert_equal_outputs(b, a)


# ---- usefulness: the residual judges a pose ---------------------------------------------------------------------------
# RMS residual per measured pixel, sqrt(SSR / (nvis * novals)), at the tracked pose: tracks against a frame of another
# scene must exceed every converged track against its true partner by this factor.  Measured on one B200: converged
# tracks at most 0.34 grey levels, unrelated ones at least 32.8, a margin of 96x; the gate leaves a factor ~10 of that.
SEPARATION = 10.0


def test_residual_separates_good_and_bad_poses(ict):
    w, h, T, n = 640, 480, 48, 100
    sc, A, B, p_gt = synth.make_pair(61, w, h)
    _, U, _, _ = synth.make_pair(62, w, h)                      # another scene: nothing to align with
    fr = ict.Frames(3, w, h, 3, 8)
    fr.upload(0, np.stack([A, B, U]))
    op = ict.make_optparam(lv_f=3, psz=8, maxiter=20, maxpttrack=n)
    tr = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
    tr.set_points(np.arange(T + 1, dtype=np.int64) * n, np.concatenate([sc.points(700 + t, n, 8, 3) for t in range(T)]))
    p0 = np.zeros((T, 6))
    rms = {}
    for name, nf in (("true", 1), ("unrelated", 2)):
        p = tr.track_batch(fr, 0, nf, p0)["p_out"]
        at = tr.evaluate(fr, 0, nf, p0, p, 0)
        start = tr.evaluate(fr, 0, nf, p0, None, 0)
        rms[name] = np.sqrt(at["ssr"] / np.maximum(at["nvis"] * op.novals, 1))
        if name == "true":
            conv = np.abs(p - p_gt).max(1) < 5e-3
            assert conv.sum() >= T // 2, conv.sum()
            assert (at["ssr"][conv] < start["ssr"][conv]).all()
    tr.close()
    fr.close()
    margin = rms["unrelated"].min() / rms["true"][conv].max()
    print("RMS per pixel: converged max %.3f, unrelated min %.3f, margin %.1fx"
          % (rms["true"][conv].max(), rms["unrelated"].min(), margin))
    assert margin > SEPARATION, margin
