"""ict_track_evaluate_poses on the GPU: K candidate poses per track against one template.

  * for every k the outputs of candidate k are those of ict_track_evaluate at p_cur = candidate k, bit for bit, and H is
    evaluate's H: every EVAL_CASES case, every level, all four sum orders, K = 1, 3 and 17 (p_ref itself, a pose that
    moves part of the points out of the new image, one that moves all of them out, small perturbations);
  * orders 1 and 3 equal the CPU model (tests/evaluate_model.py) at each candidate;
  * a candidate's outputs do not depend on K, on its position among the K or on the order of the tracks;
  * K = 256 on 32x32 tracks of the benchmark geometry, K = 4 on dense psz 1 (several tree chunks, long chains);
  * the documented errors; no side effects on later tracking calls, the 2-D points or the keep_state arrays;
  * scoring a grid of starting poses and tracking from the best one recovers motions that tracking from 0 does not.
"""
import ctypes as C

import numpy as np
import pytest

from invcompcamtrack_b200 import synth
from test_gpu_evaluate import EVAL_CASES, oracle_eval
from test_gpu_mixed_batches import G8, G32, NFR, TC, store, make_mixed, permuted, new_tracker, gpu_mixed

pytestmark = pytest.mark.gpu

FAST, SSE, GENERAL, AVX = 0, 1, 2, 3
ORDERS = (FAST, SSE, GENERAL, AVX)
OUT = ("jtr", "dp", "ssr", "nvis")


def candidates(c, K, seed):
    """[T, K, 6]: p_in, a pan that moves part of the points out of the new image, one past its width, then small
    perturbations of p_in (so the first 1 and 3 of K = 17 are the K = 1 and K = 3 sets)."""
    rng = np.random.default_rng(seed)
    T = c["T"]
    out = np.repeat(c["p_in"][:, None, :], K, 1)
    if K > 1:
        out[:, 1, 0] += 2.0
    if K > 2:
        out[:, 2, 0] += 8.0
    if K > 3:
        out[:, 3:] += np.concatenate([rng.uniform(-0.004, 0.004, (T, K - 3, 3)),
                                      rng.uniform(-0.001, 0.001, (T, K - 3, 3))], 2)
    return out


def eval_each(tr, fr, c, level, cand, ks=None):
    """ict_track_evaluate at each candidate k (all of them, or ks)."""
    ks = range(cand.shape[1]) if ks is None else ks
    return {k: tr.evaluate(fr, c["rf"], c["nf"], c["p_in"], np.ascontiguousarray(cand[:, k]), level) for k in ks}


def assert_poses_equal_evaluate(g, each, what=""):
    for k, e in each.items():
        assert np.array_equal(g["H"], e["H"], equal_nan=True), (what, k, "H")
        for name in OUT:
            assert np.array_equal(g[name][:, k], e[name], equal_nan=True), (what, k, name)


# ---- 1. equals evaluate, bit for bit -------------------------------------------------------------------------------
@pytest.mark.parametrize("geom,sizes,kw", EVAL_CASES)
def test_equals_evaluate(ict, orc, geom, sizes, kw):
    st = store(ict, orc, *geom)
    c = make_mixed(ict, st, sizes, seed=300 + sum(sizes) % 97, **kw)
    for order in ORDERS:
        tr = new_tracker(ict, c, order)
        try:
            for level in range(c["op"].lv_l, c["op"].lv_f + 1):
                cand = candidates(c, 17, 10 * level + order)
                each = eval_each(tr, st["fr"], c, level, cand)
                for K in (1, 3, 17):
                    g = tr.evaluate_poses(st["fr"], c["rf"], c["nf"], c["p_in"], cand[:, :K], level)
                    assert g["jtr"].shape == (c["T"], K, 6) and g["ssr"].shape == (c["T"], K)
                    assert_poses_equal_evaluate(g, {k: each[k] for k in range(K)}, (order, level, K))
                if not c["op"].donorm:
                    assert (g["nvis"][:, 2] == 0).all()
        finally:
            tr.close()


# ---- 2. against the CPU model directly -----------------------------------------------------------------------------
@pytest.mark.parametrize("geom,sizes,kw", [
    pytest.param(G8, [1, 7, 129, 40, 0], dict(dopatchnorm=1), id="psz8-patchnorm"),
    pytest.param(G32, [0, 1, 2, 4, 9, 13], {}, id="psz32"),
])
def test_against_model(ict, orc, geom, sizes, kw):
    st = store(ict, orc, *geom)
    c = make_mixed(ict, st, sizes, seed=77 + len(sizes), **kw)
    level = c["op"].lv_l + 1
    cand = candidates(c, 4, 5)
    for order, mode in ((SSE, 0), (AVX, 1)):
        tr = new_tracker(ict, c, order)
        try:
            g = tr.evaluate_poses(st["fr"], c["rf"], c["nf"], c["p_in"], cand, level)
        finally:
            tr.close()
        for k in range(cand.shape[1]):
            o = oracle_eval(orc, c, level, np.ascontiguousarray(cand[:, k]), mode)
            assert np.array_equal(g["H"], o["H"], equal_nan=True), (order, k)
            for name in OUT:
                assert np.array_equal(g[name][:, k], o[name], equal_nan=True), (order, k, name)


# ---- 3. independence of K, position and track order ----------------------------------------------------------------
def test_independent_of_k_position_and_track_order(ict, orc):
    st = store(ict, orc, *G8)
    c = make_mixed(ict, st, [0, 1, 3, 13, 64, 100, 129], seed=17)
    level = 1
    cand = candidates(c, 17, 3)
    perm_k = np.random.default_rng(4).permutation(17)
    perm_t = np.roll(np.arange(c["T"]), 3)
    cp = permuted(c, perm_t)
    for order in ORDERS:
        tr = new_tracker(ict, c, order)
        try:
            g = tr.evaluate_poses(st["fr"], c["rf"], c["nf"], c["p_in"], cand, level)
            shuffled = tr.evaluate_poses(st["fr"], c["rf"], c["nf"], c["p_in"], cand[:, perm_k], level)
            five = tr.evaluate_poses(st["fr"], c["rf"], c["nf"], c["p_in"], cand[:, 6:11], level)
        finally:
            tr.close()
        trp = new_tracker(ict, cp, order)
        try:
            gp = trp.evaluate_poses(st["fr"], cp["rf"], cp["nf"], cp["p_in"], cand[perm_t], level)
        finally:
            trp.close()
        assert np.array_equal(gp["H"], g["H"][perm_t], equal_nan=True), order
        for name in OUT:
            assert np.array_equal(shuffled[name], g[name][:, perm_k], equal_nan=True), (order, name, "position")
            assert np.array_equal(five[name], g[name][:, 6:11], equal_nan=True), (order, name, "K")
            assert np.array_equal(gp[name], g[name][perm_t], equal_nan=True), (order, name, "tracks")


# ---- 4. large K, large tracks --------------------------------------------------------------------------------------
def test_large_k_on_psz32_tracks(ict):
    w, h, T, K = 1920, 1080, 64, 256
    sc, A, B, _ = synth.make_pair(91, w, h)
    fr = ict.Frames(2, w, h, 3, 32)
    fr.upload(0, np.stack([A, B]))
    op = ict.make_optparam(lv_f=3, psz=32, maxiter=10, maxpttrack=4)
    rng = np.random.default_rng(8)
    cand = np.concatenate([rng.uniform(-0.05, 0.05, (T, K, 3)), rng.uniform(-0.01, 0.01, (T, K, 3))], 2)
    c = dict(rf=np.zeros(T, np.int32), nf=np.ones(T, np.int32), p_in=np.zeros((T, 6)))
    for order in (SSE, FAST):
        tr = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
        tr.set_sum_order(order)
        tr.set_points(np.arange(T + 1, dtype=np.int64) * 4, np.concatenate([sc.points(7000 + t, 4, 32, 3) for t in range(T)]))
        try:
            for level in (0, 3):
                g = tr.evaluate_poses(fr, 0, 1, c["p_in"], cand, level)
                assert_poses_equal_evaluate(g, eval_each(tr, fr, c, level, cand, (0, 1, 100, 254, 255)), (order, level))
                assert (g["nvis"] > 0).mean() > 0.5
        finally:
            tr.close()
    fr.close()


@pytest.mark.parametrize("donorm", [0, 1])
def test_dense_tracks(ict, orc, donorm):
    st = store(ict, orc, 1, 320, 240, 2)
    c = make_mixed(ict, st, [8, 0, 1], seed=5, donorm=donorm, dense=0)
    assert c["sizes"][0] > 4096          # several tree-order chunks, long reference-order chains
    cand = candidates(c, 4, 6)
    for order in ORDERS:
        tr = new_tracker(ict, c, order)
        try:
            g = tr.evaluate_poses(st["fr"], c["rf"], c["nf"], c["p_in"], cand, 0)
            assert_poses_equal_evaluate(g, eval_each(tr, st["fr"], c, 0, cand), (order, donorm))
        finally:
            tr.close()


# ---- 5. errors and side effects ------------------------------------------------------------------------------------
def test_errors(ict, orc):
    st = store(ict, orc, *G8)
    c = make_mixed(ict, st, [5, 9], seed=41)
    tr = new_tracker(ict, c, SSE)
    cand = candidates(c, 3, 1)

    def ev(rf=c["rf"], level=None, p_cand=cand):
        return tr.evaluate_poses(st["fr"], rf, c["nf"], c["p_in"], p_cand, level)

    for bad in (dict(level=c["op"].lv_f + 1), dict(level=c["op"].lv_l - 1), dict(rf=np.array([0, NFR])),
                dict(p_cand=cand[:, :0])):
        with pytest.raises(ict.IctError, match="ICT_ERR_BAD_ARG"):
            ev(**bad)
    lib = ict.lib()
    rf, nf = np.ascontiguousarray(c["rf"], np.int32), np.ascontiguousarray(c["nf"], np.int32)
    p_ref = np.ascontiguousarray(c["p_in"])
    ptr = lambda a: C.c_void_p(a.ctypes.data)  # noqa: E731
    for K, p in ((3, None), (2 ** 30, ptr(cand))):       # NULL p_cand; T*K = 2^31 beyond INT_MAX
        rc = lib.ict_track_evaluate_poses(tr.h_, st["fr"].h_, ptr(rf), ptr(nf), ptr(p_ref), K, p, 0, None, None, None,
                                          None, None)
        assert rc == 2, (K, rc)
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


def test_no_side_effects(ict, orc):
    st = store(ict, orc, *G8)
    c = make_mixed(ict, st, [0, 1, 13, 64, 100], seed=31)
    cand = candidates(c, 5, 2)
    for order in (SSE, FAST):
        ref = gpu_mixed(ict, c, order)
        tr = new_tracker(ict, c, order)
        tr.evaluate_poses(st["fr"], c["rf"], c["nf"], c["p_in"] * 0.5, cand, 1)
        out = tr.track_batch(st["fr"], c["rf"], c["nf"], c["p_in"], trace_cap=TC)
        out["pt2d"] = tr.get_2dpoints()
        tr.evaluate_poses(st["fr"], c["nf"], c["rf"], c["p_in"], cand, 0)
        assert np.array_equal(tr.get_2dpoints(), out["pt2d"])
        tr.close()
        for k in ("p_out", "iters", "npixres", "pt2d"):
            assert np.array_equal(out[k], ref[k], equal_nan=True), (order, k)
        assert np.array_equal(out["trace"][..., :16], ref["trace"][..., :16], equal_nan=True)
    runs = []
    for with_eval in (False, True):
        tr = new_tracker(ict, c, SSE, knobs=(("keep_state", 1),))
        p = c["p_in"]
        poses = []
        for k in range(3):
            if with_eval:
                tr.evaluate_poses(st["fr"], np.full(c["T"], k + 1), np.full(c["T"], k), p, cand, 2)
            p = tr.track_batch(st["fr"], np.full(c["T"], k), np.full(c["T"], k + 1), p)["p_out"]
            poses.append(p)
        tr.close()
        runs.append(np.stack(poses))
    assert np.array_equal(runs[0], runs[1], equal_nan=True)


# ---- 6. usefulness: multi-start for motions beyond the pyramid's basin ---------------------------------------------
MOTION_SCALE = 6.0        # random_motion's default scaled 6x: image flow up to ~80 px at level 0
GN_ITERS = 12             # Gauss-Newton updates per level


def start_grid():
    """Starting poses around 0: a 5x5 grid of x / y translations, translations along and rotations about the optical
    axis (33 poses; an x / y translation moves the image like a rotation about the other axis)."""
    g = [np.array([tx, ty, 0, 0, 0, 0.0]) for tx in (-0.5, -0.25, 0, 0.25, 0.5) for ty in (-0.5, -0.25, 0, 0.25, 0.5)]
    for a in (-0.3, -0.15, 0.15, 0.3):
        g.append(np.array([0, 0, a, 0, 0, 0.0]))
    for a in (-0.06, -0.03, 0.03, 0.06):
        g.append(np.array([0, 0, 0, 0, 0, a]))
    return np.array(g)


def multistart_counts(ict, seeds, T=32, n=100):
    """Tracks (over the seeds' pairs) that converge to p_gt from 0 and from the start of start_grid with the lowest RMS
    residual per measured pixel at lv_f.  Both starts run TrackPose's update p += dp (odometer.cpp:407-410) from
    lv_f down to lv_l, GN_ITERS times per level, as two candidates of one evaluate_poses call per iteration."""
    w, h = 640, 480
    grid = start_grid()
    from0 = best = total = 0
    for seed in seeds:
        sc, A, B, p_gt = synth.make_pair(seed, w, h, motion_scale=MOTION_SCALE)
        fr = ict.Frames(2, w, h, 3, 8)
        fr.upload(0, np.stack([A, B]))
        op = ict.make_optparam(lv_f=3, psz=8, maxiter=20, maxpttrack=n)
        tr = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
        tr.set_points(np.arange(T + 1, dtype=np.int64) * n,
                      np.concatenate([sc.points(900 + t, n, 8, 3) for t in range(T)]))
        p0 = np.zeros((T, 6))
        try:
            s = tr.evaluate_poses(fr, 0, 1, p0, grid[None], op.lv_f)
            rms = np.sqrt(s["ssr"] / np.maximum(s["nvis"] * op.novals, 1))
            rms[s["nvis"] == 0] = np.inf
            p = np.stack([p0, grid[np.argmin(rms, 1)]], 1)          # [T, 2, 6]: from 0, from the best start
            for level in range(op.lv_f, op.lv_l - 1, -1):
                for _ in range(GN_ITERS):
                    p = p + tr.evaluate_poses(fr, 0, 1, p0, p, level)["dp"]
        finally:
            tr.close()
            fr.close()
        ok = np.abs(p - p_gt).max(2) < 5e-3
        from0 += int(ok[:, 0].sum())
        best += int(ok[:, 1].sum())
        total += T
    return from0, best, total


# Measured on one B200 at a 1000 W power limit (seeds 71-74, 128 tracks, motion 6x the default): 62 tracks converge from
# 0 and 124 from the best start (48 % and 97 %).  The gates leave a margin of about 20 points of share on each side.
USEFUL_SEEDS = (71, 72, 73, 74)


def test_multistart_recovers_large_motion(ict):
    from0, best, total = multistart_counts(ict, USEFUL_SEEDS)
    print("converged from 0: %d / %d, from the best start: %d / %d" % (from0, total, best, total))
    assert from0 <= 0.7 * total, from0            # the motion is beyond the basin for a clear share of the tracks
    assert best >= from0 + 0.3 * total, (from0, best)
