"""ict_track_batch_from: SetPose at p_ref, TrackPose from p_start, on every tracking kernel.

The rows are those of tests/test_gpu_replay.py (every kernel family, both multi-CTA dense forms, every sum order).

  * identity: no p_start, or p_start = p_ref, returns the bits of ict_track_batch in every output (p_out, iters,
    npixres, the trace records, the 2-D points) and launches as many kernels;
  * replay: from a start pose of its own per track, each traced iteration is measured again by the CPU model
    (tests/evaluate_model.py), whose template depends on p_ref only and whose trajectory starts at p_start: exact
    trajectory checks, p_out = the rebuilt final pose, nvis equal up to points at the bounds; orders 1 and 3 bit for
    bit, orders 0 and 2 within gates measured on the B200; the untraced call returns the same bits and the call
    runs the kernels ict_track_batch runs;
  * the first record of a reference-order run is ict_track_evaluate(p_ref, p_cur = p_start) at lv_f;
  * keep_state carries a template that does not depend on the start; the device form on a stream; non-finite start
    rows; errors;
  * ground truth: beyond the pyramid's basin, tracking from a prediction near the true pose converges where tracking
    from the reference pose does not.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from invcompcamtrack_b200 import api, synth
from helpers import replay_models, check_trajectory, replay_trace_cap, teacher_forced_errors
from evaluate_model import replay_batch
from test_gpu_kernel_routing import kernels_of
from test_gpu_replay import ROWS, build_case, ORACLE_MODE, FAST, SSE, AVX

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT_KEYS = ("p_out", "iters", "npixres", "trace")

# Gates of the replay from a start pose in orders 0 and 2: (J^T r relative to sum|sd_k * pdiff|, delta_p relative to
# the level's first step), the worst values measured on one NVIDIA B200 at its 1000 W power limit x 3 (DESIGN.md §5).
FROM_GATES = {
    "v8-8w-lvl1": (1.7e-6, 2.6e-3),
    "v8-16w-motion": (1.9e-6, 7.7e-3),
    "v8-8w-pn": (4.8e-5, 1.6e-3),
    "v8-16w-pn-cap": (1.4e-5, 7.5e-3),
    "v8-8w-donorm-pn": (2.3e-5, 1.1e-2),
    "fast8-250": (1.4e-6, 8.6e-3),
    "fast16-9-donorm": (1.3e-4, 5.2e-2),
    "fast16-70": (1.7e-6, 1.6e-2),
    "fast32-18": (1.2e-6, 6.1e-3),
    "v2-4-onept": (2.5e-5, 1.4e-1),
    "v2-8": (3.8e-6, 2.4e-2),
    "v2-16-lvl1": (2.5e-6, 1.5e-2),
    "general-psz4": (4.6e-7, 9.5e-4),
    "general-psz7-pn": (7.7e-5, 1.6e-3),
    "general-psz16-pn": (4.6e-5, 7.4e-3),
    "general-psz32-pn": (7.4e-5, 4.8e-2),
    "multi-psz8-300": (1.1e-6, 4.2e-3),
    "multi-psz8-242-pn": (8.3e-6, 6.6e-3),
    "multi-psz16-71": (1.5e-6, 1.4e-2),
    "multi-psz32-19": (4.6e-7, 7.8e-3),
    "dense-tma": (5.9e-7, 1.5e-4),
    "dense-ldg": (4.2e-7, 3.3e-4),
    "o2-general-psz8": (9.2e-7, 3.5e-3),
    "o2-general-psz8-pn": (1.9e-5, 4.8e-3),
    "o2-general-psz16": (1.3e-6, 7.7e-3),
    "o2-general-psz32": (1.3e-6, 2.8e-2),
    "o2-multi-psz1": (4.2e-7, 1.5e-4),
}


def open_case(ict, c, order, knobs=(), robust=0, nframes=2):
    op = ict.OptParam.from_buffer_copy(bytes(c["op"]))
    fr = ict.Frames(nframes, c["w"], c["h"], c["lv_f"], c["psz"])
    tr = ict.Tracker(op, c["sc"].fc, c["sc"].cc, c["sc"].wh)
    fr.upload(0, np.stack([c["A"], c["B"]] * (nframes // 2)))
    tr.set_sum_order(order)
    for k, v in knobs:
        tr.set_knob(k, v)
    if robust:
        tr.set_robust(robust)
    tr.set_points(c["pt_off"], c["pts"].copy())
    return tr, fr


def track_from_null(tr, fr, p_ref, cap):
    """ict_track_batch_from with p_start = NULL (Tracker.track_batch calls ict_track_batch for that)."""
    T, L = tr.T, tr.L
    rf, nf = np.zeros(T, np.int32), np.ones(T, np.int32)
    p_ref = np.ascontiguousarray(np.broadcast_to(p_ref, (T, 6)), np.float64)
    out = dict(p_out=np.zeros((T, 6)), iters=np.zeros((T, L), np.int32), npixres=np.zeros(T, np.int64),
               trace=np.zeros((T, cap, api.TRACE_FLOATS), np.float32) if cap else None)
    api._check(api.lib().ict_track_batch_from(tr.h_, fr.h_, api._p(rf), api._p(nf), api._p(p_ref), None,
                                              api._p(out["p_out"]), api._p(out["iters"]), api._p(out["trace"]), cap,
                                              api._p(out["npixres"])))
    return out


def same_bits(a, b, keys=OUT_KEYS):
    """Bit equality of the outputs; of the trace, fields 0-15 (16-23 hold the SM cycle counts some kernels record)."""
    for k in keys:
        x, y = a[k], b[k]
        assert (x is None) == (y is None), k
        if x is not None and k == "trace":
            x, y = x[..., :16], y[..., :16]
        if x is not None:
            assert x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes(), k


def start_poses(c, p_ref, r):
    """A start pose per track: p_ref plus a distinct offset of up to ~6 px of image motion at level 0, track 0 left at
    p_ref when there are several (a kernel that reads another track's row is caught).  With edge points (last track)
    that track moves ~8 px along x, so that points near the left or right border start across the bounds."""
    T = c["T"]
    s = 640.0 / c["w"]
    rng = np.random.default_rng(7000 + r["kw"]["seed"])
    off = np.concatenate([rng.uniform(-0.05, 0.05, (T, 3)), rng.uniform(-0.004, 0.004, (T, 3))], 1) * s
    if r["edge"]:
        off[-1, 0] = 0.06 * s * (1 if r["kw"]["seed"] % 2 else -1)
    if T > 1:
        off[0] = 0.0
    return p_ref + off


# ---- 1. identity ---------------------------------------------------------------------------------------------------
def identity_calls(ict, tr, fr, p_ref, cap):
    """ict_track_batch, ict_track_batch_from(p_start = NULL), ict_track_batch_from(p_start = p_ref): outputs with the
    2-D points, and the launches of each call."""
    res = []
    for call in (lambda: tr.track_batch(fr, 0, 1, p_ref, trace_cap=cap),
                 lambda: track_from_null(tr, fr, p_ref, cap),
                 lambda: tr.track_batch(fr, 0, 1, p_ref, trace_cap=cap, p_start=p_ref.copy())):
        n0 = ict.launch_count()
        out = call()
        out["launches"] = ict.launch_count() - n0
        out["pt2d"] = tr.get_2dpoints()
        res.append(out)
    return res


def check_identity(res):
    for other in res[1:]:
        same_bits(res[0], other, OUT_KEYS + ("pt2d",))
        assert other["launches"] == res[0]["launches"], (other["launches"], res[0]["launches"])


@pytest.mark.gpu
@pytest.mark.parametrize("r", ROWS)
def test_identity(ict, r):
    c, p_ref = build_case(r)
    tr, fr = open_case(ict, c, r["order"])
    try:
        check_identity(identity_calls(ict, tr, fr, p_ref, replay_trace_cap(c["op"])))
        check_identity(identity_calls(ict, tr, fr, p_ref, 0))
    finally:
        tr.close()
        fr.close()


def small_case(**kw):
    from helpers import make_case
    return make_case(**dict(dict(seed=451, psz=8, npts=100, ntracks=3), **kw))


@pytest.mark.gpu
def test_identity_keep_state(ict):
    """K2x8 (100 points of 8x8, reference order: the only kernel with keep_state) with the carried template: two
    successive calls of each form give the same bits."""
    c = small_case()
    p_ref = np.zeros((c["T"], 6))
    cap = replay_trace_cap(c["op"])
    runs = []
    for form in range(3):
        tr, fr = open_case(ict, c, SSE, knobs=(("keep_state", 1),))
        try:
            calls = []
            for _ in range(2):
                if form == 0:
                    out = tr.track_batch(fr, 0, 1, p_ref, trace_cap=cap)
                elif form == 1:
                    out = track_from_null(tr, fr, p_ref, cap)
                else:
                    out = tr.track_batch(fr, 0, 1, p_ref, trace_cap=cap, p_start=p_ref)
                out["pt2d"] = tr.get_2dpoints()
                calls.append(out)
            runs.append(calls)
        finally:
            tr.close()
            fr.close()
    for form in (1, 2):
        for k in range(2):
            same_bits(runs[0][k], runs[form][k], OUT_KEYS + ("pt2d",))


@pytest.mark.gpu
@pytest.mark.parametrize("flag", [api.ROBUST_FULL_STEP, api.ROBUST_COMPOSE, api.ROBUST_FLOOR])
def test_identity_robust(ict, flag):
    """K2v8 (100 points of 8x8, fast mode: the only kernel with the robustness flags) under each flag."""
    c = small_case(seed=452)
    p_ref = np.zeros((c["T"], 6))
    tr, fr = open_case(ict, c, FAST, robust=flag)
    try:
        check_identity(identity_calls(ict, tr, fr, p_ref, replay_trace_cap(c["op"])))
    finally:
        tr.close()
        fr.close()


# ---- 2. replay from another start ----------------------------------------------------------------------------------
def run_from(ict, c, p_ref, p_start, order, cap, profile=False):
    """The from-call untraced and traced (and, with profile, the names of the kernels that each of track_batch
    untraced, traced and the two from-calls launched)."""
    tr, fr = open_case(ict, c, order)
    try:
        calls = (lambda: tr.track_batch(fr, 0, 1, p_ref, p_start=p_start),
                 lambda: tr.track_batch(fr, 0, 1, p_ref, trace_cap=cap, p_start=p_start))
        if profile:
            plain = (lambda: tr.track_batch(fr, 0, 1, p_ref), lambda: tr.track_batch(fr, 0, 1, p_ref, trace_cap=cap))
            return [kernels_of(f) for f in plain + calls]
        return calls[0](), calls[1](), (fr.download(0), fr.download(1))
    finally:
        tr.close()
        fr.close()


def profile_rows(path):
    """{row id: [track_batch untraced, traced, from-call untraced, traced] kernel names} for every row (JSON)."""
    import invcompcamtrack_b200 as ict
    ict.lib()
    out = {}
    for p in ROWS:
        r = p.values[0]
        c, p_ref = build_case(r)
        out[p.id] = run_from(ict, c, p_ref, start_poses(c, p_ref, r), r["order"], replay_trace_cap(c["op"]),
                             profile=True)
    with open(path, "w") as f:
        json.dump(out, f)


@pytest.fixture(scope="module")
def from_kernels(tmp_path_factory):
    """The kernels of every row, profiled in a fresh process (see test_gpu_replay.row_kernels)."""
    path = str(tmp_path_factory.mktemp("from") / "kernels.json")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, HERE, os.environ.get("PYTHONPATH", "")]))
    r = subprocess.run([sys.executable, "-c", "import test_gpu_track_from as m, sys; m.profile_rows(sys.argv[1])",
                        path], cwd=HERE, env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    with open(path) as f:
        return json.load(f)


def replay_from(orc, c, pyr, p_ref, p_start, g, order):
    models = replay_models(orc, c, pyr, p_ref)
    for t, m in enumerate(models):
        m.p0 = m.internal(p_start[t])
    orc.set_sum_mode(ORACLE_MODE[order])
    try:
        return replay_batch(models, g["trace"])
    finally:
        orc.set_sum_mode(0)


@pytest.mark.gpu
@pytest.mark.parametrize("r", ROWS)
def test_replay_from(ict, orc, from_kernels, request, r):
    c, p_ref = build_case(r)
    p_start = start_poses(c, p_ref, r)
    op, order = c["op"], r["order"]
    names = from_kernels[request.node.callspec.id]
    assert names[2] == names[0] and names[3] == names[1], names
    g0, g, pyr = run_from(ict, c, p_ref, p_start, order, replay_trace_cap(op))

    check_trajectory(g, op)
    rep = replay_from(orc, c, pyr, p_ref, p_start, g, order)
    m = rep["trace"]
    assert np.array_equal(g["p_out"], rep["p_out"]), (g["p_out"], rep["p_out"])
    nflip = 0
    for t in range(c["T"]):
        n = int((g["trace"][t, :, 0] >= 0).sum())
        d = np.abs(g["trace"][t, :n, 15].astype(np.int64) - m[t, :n, 15].astype(np.int64))
        assert (d <= rep["nborder"][t]).all(), (t, np.flatnonzero(d > rep["nborder"][t]))
        nflip += int(d.sum())
    if order in (SSE, AVX):
        assert np.array_equal(g["trace"][..., :16], m[..., :16])
        msg = "bit-identical"
    else:
        jtr, dp, _ = teacher_forced_errors(g, dict(trace=m))
        jtr_tol, dp_tol = FROM_GATES[request.node.callspec.id]
        msg = "J^T r %.2e of sum|sd*r| (gate %.1e), delta_p %.2e of the level's first step (gate %.1e)" % (
            jtr, jtr_tol, dp, dp_tol)
        assert jtr <= jtr_tol and dp <= dp_tol, msg
    print("from %s: %s, %d records, %d nvis flips at the bounds, levels %s" % (
        request.node.callspec.id, msg, int((g["trace"][..., 0] >= 0).sum()), nflip, g["iters"].tolist()))
    for k in ("p_out", "iters", "npixres"):
        assert np.array_equal(g0[k], g[k]), k


# ---- 3. the first record is ict_track_evaluate at the start pose -----------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("r", [p for p in ROWS if p.values[0]["order"] in (SSE, AVX)])
def test_first_record_is_evaluate(ict, r):
    c, p_ref = build_case(r)
    p_start = start_poses(c, p_ref, r)
    lv_f = c["op"].lv_f
    tr, fr = open_case(ict, c, r["order"])
    try:
        g = tr.track_batch(fr, 0, 1, p_ref, trace_cap=replay_trace_cap(c["op"]), p_start=p_start)
        ev = tr.evaluate(fr, 0, 1, p_ref, p_cur=p_start, level=lv_f)
    finally:
        tr.close()
        fr.close()
    first = g["trace"][:, 0]
    assert (first[:, 0] == lv_f).all() and (first[:, 1] == 0).all()
    assert first[:, 2:8].tobytes() == ev["jtr"].tobytes()
    assert first[:, 8:14].tobytes() == ev["dp"].tobytes()
    assert np.array_equal(first[:, 15].astype(np.int32), ev["nvis"])


# ---- 4. the carried template does not depend on the start ------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("order", [SSE, AVX])
def test_keep_state_after_from(ict, order):
    c = small_case(seed=453)
    p_ref = np.zeros((c["T"], 6))
    p_start = start_poses(c, p_ref, dict(kw=dict(seed=453), edge=0))
    cap = replay_trace_cap(c["op"])
    second = []
    for first_start in (p_start, None):
        tr, fr = open_case(ict, c, order, knobs=(("keep_state", 1),))
        try:
            tr.track_batch(fr, 0, 1, p_ref, trace_cap=cap, p_start=first_start)
            out = tr.track_batch(fr, 0, 1, p_ref, trace_cap=cap)
            out["pt2d"] = tr.get_2dpoints()
            second.append(out)
        finally:
            tr.close()
            fr.close()
    same_bits(second[0], second[1], OUT_KEYS + ("pt2d",))


# ---- 5. forms and errors -------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("order", [FAST, SSE])
def test_device_form_on_stream(ict, order):
    import torch
    c = small_case(seed=454)
    T = c["T"]
    p_ref = np.zeros((T, 6))
    p_start = start_poses(c, p_ref, dict(kw=dict(seed=454), edge=0))
    cap = replay_trace_cap(c["op"])
    tr, fr = open_case(ict, c, order)
    try:
        want = tr.track_batch(fr, 0, 1, p_ref, trace_cap=cap, p_start=p_start)
    finally:
        tr.close()
    op = ict.OptParam.from_buffer_copy(bytes(c["op"]))
    tr = ict.Tracker(op, c["sc"].fc, c["sc"].cc, c["sc"].wh)
    try:
        tr.set_sum_order(order)
        dev = torch.device("cuda", 0)
        st = torch.cuda.Stream(device=dev)
        L = tr.L
        with torch.cuda.stream(st):
            d_off = torch.as_tensor(c["pt_off"], device=dev)
            d_pts = torch.as_tensor(c["pts"], device=dev)
            d_rf = torch.zeros(T, dtype=torch.int32, device=dev)
            d_nf = torch.ones(T, dtype=torch.int32, device=dev)
            d_ref = torch.as_tensor(p_ref, device=dev)
            d_start = torch.as_tensor(p_start, device=dev)
            d_out = torch.zeros((T, 6), dtype=torch.float64, device=dev)
            d_it = torch.zeros((T, L), dtype=torch.int32, device=dev)
            d_np = torch.zeros(T, dtype=torch.int64, device=dev)
            d_tr = torch.zeros((T, cap, api.TRACE_FLOATS), dtype=torch.float32, device=dev)
        s = st.cuda_stream
        tr.set_points_dev(T, d_off.data_ptr(), d_pts.data_ptr(), int(c["pt_off"][-1]), int(np.diff(c["pt_off"]).max()),
                          stream=s)
        tr.track_batch_dev(fr, d_rf.data_ptr(), d_nf.data_ptr(), d_ref.data_ptr(), d_out.data_ptr(), d_it.data_ptr(),
                           d_np.data_ptr(), d_tr.data_ptr(), cap, stream=s, p_start_ptr=d_start.data_ptr())
        st.synchronize()
        got = dict(p_out=d_out.cpu().numpy(), iters=d_it.cpu().numpy(), npixres=d_np.cpu().numpy(),
                   trace=d_tr.cpu().numpy())
    finally:
        tr.close()
        fr.close()
    same_bits(want, got)
    assert not np.array_equal(want["p_out"][1:], np.zeros_like(want["p_out"][1:]))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["multi-cta", "k2v8", "k2x8"])
def test_non_finite_start(ict, kind):
    """Non-finite start rows: every point starts outside the new image; the call succeeds, those tracks see no pixel,
    the other tracks are unaffected."""
    # the kernel follows from the configuration (tests/test_gpu_kernel_routing.py): 300 points of 8x8 in fast mode run
    # the multi-CTA path, 100 points K2v8 in fast mode and K2x8 in reference order
    if kind == "multi-cta":
        c, order = small_case(seed=455, npts=300, ntracks=2), FAST
    elif kind == "k2v8":
        c, order = small_case(seed=456, ntracks=4), FAST
    else:
        c, order = small_case(seed=457, ntracks=4), SSE
    T = c["T"]
    p_ref = np.zeros((T, 6))
    good = start_poses(c, p_ref, dict(kw=dict(seed=455), edge=0))
    bad = good.copy()
    bad[1] = np.nan
    if T > 2:
        bad[3, 0] = np.inf
    bad_rows = [1] + ([3] if T > 2 else [])
    cap = replay_trace_cap(c["op"])
    tr, fr = open_case(ict, c, order)
    try:
        g = tr.track_batch(fr, 0, 1, p_ref, trace_cap=cap, p_start=bad)
        ok = tr.track_batch(fr, 0, 1, p_ref, trace_cap=cap, p_start=good)
    finally:
        tr.close()
        fr.close()
    L = c["op"].lv_f - c["op"].lv_l + 1
    for t in range(T):
        if t in bad_rows:
            recs = g["trace"][t][g["trace"][t, :, 0] >= 0]
            assert len(recs) == L and (recs[:, 15] == 0).all(), recs[:, [0, 1, 15]]
            assert (g["iters"][t] == 1).all() and g["npixres"][t] == 0
            assert not np.isfinite(g["p_out"][t]).all()
        else:
            same_bits({k: g[k][t] for k in OUT_KEYS}, {k: ok[k][t] for k in OUT_KEYS})


@pytest.mark.gpu
def test_errors(ict):
    c = small_case(seed=458)
    p_ref = np.zeros((c["T"], 6))
    tr, fr = open_case(ict, c, SSE)
    other = ict.Frames(2, c["w"], c["h"], c["lv_f"] - 1, c["psz"])
    try:
        with pytest.raises(ict.IctError, match="ICT_ERR_BAD_ARG"):
            tr.track_batch(fr, 0, 2, p_ref, p_start=p_ref)
        with pytest.raises(ict.IctError, match="ICT_ERR_BAD_ARG"):
            tr.track_batch(fr, -1, 1, p_ref, p_start=p_ref)
        with pytest.raises(ict.IctError, match="ICT_ERR_BAD_ARG"):
            tr.track_batch(other, 0, 1, p_ref, p_start=p_ref)
    finally:
        other.close()
        tr.close()
        fr.close()


# ---- 6. what the feature is for ------------------------------------------------------------------------------------
GT_SCENES, GT_MOTIONS, GT_W, GT_H, GT_LV, GT_PSZ, GT_NPTS = 8, 8, 640, 480, 3, 8, 100
GT_TRACKS = GT_SCENES * GT_MOTIONS


def gt_scenes(seed0=900):
    """The textured planes of synth.make_pair for seeds seed0.., each with its frame at pose 0 and 100 points."""
    out = []
    for s in range(GT_SCENES):
        sc = synth.Scene(seed0 + s, GT_W, GT_H)
        out.append((sc, sc.render(np.zeros(6)), sc.points(seed0 + s, GT_NPTS, GT_PSZ, GT_LV)))
    return out


def gt_pairs(scenes, scale, seed0=900):
    """64 tracks, GT_MOTIONS per scene, each on a frame pair of its own: synth.make_pair's motion at `scale` (its
    random_motion, a seed per track) and the new frame rendered there.  Returns (frames, ref_frame, new_frame, points,
    p_gt): frames 0..GT_SCENES-1 are the scenes' frames at pose 0, frame GT_SCENES + t the new frame of track t."""
    frames = [A for _, A, _ in scenes]
    pts, p_gt = [], []
    for t in range(GT_TRACKS):
        sc, _, P = scenes[t // GT_MOTIONS]
        gt = sc.random_motion(seed0 + 100 + t, scale)
        frames.append(sc.render(gt))
        pts.append(P)
        p_gt.append(gt)
    rf = (np.arange(GT_TRACKS) // GT_MOTIONS).astype(np.int32)
    nf = (GT_SCENES + np.arange(GT_TRACKS)).astype(np.int32)
    return np.stack(frames), rf, nf, np.concatenate(pts), np.array(p_gt)


def gt_tracker(ict, scenes, frames, order, pts, copies=1):
    """A tracker with each track's points `copies` times (multi-start) and a frame store of `frames`."""
    sc = scenes[0][0]
    op = ict.make_optparam(lv_f=GT_LV, psz=GT_PSZ, maxiter=10, maxpttrack=GT_NPTS)
    fr = ict.Frames(len(frames), GT_W, GT_H, GT_LV, GT_PSZ)
    fr.upload(0, frames)
    tr = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
    tr.set_sum_order(order)
    per = pts.reshape(GT_TRACKS, 3 * GT_NPTS)
    tr.set_points(np.arange(GT_TRACKS * copies + 1, dtype=np.int64) * GT_NPTS, np.repeat(per, copies, 0).reshape(-1))
    return tr, fr


def gt_prediction(p_gt, frac, seed=1):
    """p_gt perturbed by up to frac of the motion in every coefficient: a prediction that is close, not exact."""
    return p_gt + frac * np.abs(p_gt) * np.random.default_rng(seed).uniform(-1, 1, p_gt.shape)


def gt_error(p_out, p_gt):
    return np.abs(p_out - p_gt).max(1)


# Motion scale, tolerance on |p_out - p_gt|_inf and perturbation of the prediction, from the basin table of
# profiles/tools/from_time.py (DESIGN.md §6), measured on the B200.
GT_SCALE, GT_TOL, GT_FRAC = 8.0, 5e-2, 0.1


@pytest.fixture(scope="module")
def gt_case():
    scenes = gt_scenes()
    return scenes, gt_pairs(scenes, GT_SCALE)


@pytest.mark.gpu
@pytest.mark.parametrize("order", [SSE, FAST])
def test_ground_truth_beyond_the_basin(ict, gt_case, order):
    scenes, (frames, rf, nf, pts, p_gt) = gt_case
    tr, fr = gt_tracker(ict, scenes, frames, order, pts)
    try:
        zero = np.zeros((GT_TRACKS, 6))
        e_ref = gt_error(tr.track_batch(fr, rf, nf, zero)["p_out"], p_gt)
        e_pred = gt_error(tr.track_batch(fr, rf, nf, zero, p_start=gt_prediction(p_gt, GT_FRAC))["p_out"], p_gt)
    finally:
        tr.close()
        fr.close()
    off_ref, ok_pred = int((e_ref > GT_TOL).sum()), int((e_pred <= GT_TOL).sum())
    print("motion scale %g: from p_ref %d/%d tracks off p_gt, from the prediction %d/%d on it" % (
        GT_SCALE, off_ref, GT_TRACKS, ok_pred, GT_TRACKS))
    # measured on the B200: 53 of 64 off from p_ref, 64 of 64 on from the prediction (worst error 0.027), both orders
    assert off_ref >= GT_TRACKS // 2
    assert ok_pred >= GT_TRACKS - 2
