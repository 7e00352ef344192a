"""Every iteration of every tracking kernel, checked against a CPU replay of the kernel's own trajectory.

A traced ict_track_batch records per iteration the level, J^T r, delta_p, normdp and the visible points.  Every kernel
updates its fp32 pose coefficients additively with the delta_p it records, so the pose at which it took each measurement
is rebuilt exactly from p_in and the trace, and the CPU model (tests/evaluate_model.py, pinned to the oracle by
tests/test_oracle_replay.py) measures again at that pose.  Per row, the kernel is pinned by name (the routing table of
tests/test_gpu_kernel_routing.py, traced and untraced), and then:

  * in every sum order, exactly: the records' level / iteration structure, iters, the stop rule on the kernel's own
    normdp, normdp = |delta_p|_1, npixres = novals * sum nvis (helpers.check_trajectory); p_out = getPose_se3 of the
    rebuilt final pose; every record's nvis equals the model's, except for points within 1e-3 px of the image bounds;
  * orders 1 and 3 (reference summation orders): every record bit-identical to the replay in the oracle's sum mode
    0 / 1;
  * orders 0 and 2 (tree sums): J^T r within 1e-5 of sum_k |sd_k * pdiff| on every record, the gate
    test_jtr_teacher_forced applies, here on the kernel's own trajectory; delta_p within the row's gate, relative to the
    level's first step (helpers.teacher_forced_errors); the untraced run returns the same p_out / iters / npixres bits.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import make_case, replay_models, check_trajectory, replay_trace_cap, teacher_forced_errors
from evaluate_model import replay_batch
from test_gpu_kernel_routing import kernels_of, assert_routed, MULTI, DENSE_TMA, DENSE_LDG

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
FAST, SSE, GENERAL, AVX = 0, 1, 2, 3
ORACLE_MODE = {FAST: 0, SSE: 0, GENERAL: 0, AVX: 1}       # the oracle's sum mode each order is replayed in
P_START = [0.01, -0.02, 0.005, 0.002, -0.001, 0.003]      # a start pose other than 0, through donorm's normalisation
G8, G16, G32, G1 = dict(w=640, h=480, lv_f=3), dict(w=960, h=544, lv_f=3), dict(w=1920, h=1080, lv_f=3), \
    dict(w=320, h=240, lv_f=2)


def row(rid, order, want, dp_tol=None, jtr_tol=1e-5, sizes=None, edge=0, p_in=None, **kw):
    """rid: test id; want: the kernel as the routing table names it (untraced); dp_tol, jtr_tol: the delta_p and J^T r
    gates of orders 0 / 2 (see ROWS); sizes: points per track (else ntracks x npts); edge: that many points of
    the last track within 6 px of the left or right image border, so that they leave and re-enter the new frame during
    the first level; p_in: the start pose of every track; kw: make_case options."""
    return pytest.param(dict(order=order, want=want, dp_tol=dp_tol, jtr_tol=jtr_tol, sizes=sizes, edge=edge, p_in=p_in,
                             kw=kw), id=rid)


# Gates of orders 0 and 2, measured on one NVIDIA B200 at its 1000 W power limit, x 3 (DESIGN.md §5 item 2 lists the
# measured values).  delta_p: worst error relative to the level's first step.  J^T r: 1e-5 of sum|sd_k * pdiff| except
# in the five dopatchnorm rows that measured above it (1.4e-5 .. 2.6e-5).  There every pixel difference carries the
# fp32 rounding of its two patch means, which a tree sum and Eigen's packet order round differently; that error scales
# with the intensities, not with pdiff, so near convergence sum|sd_k * pdiff| understates it.  The oracle itself moves
# as much when only its sum order changes: replayed along the same trajectories in its sum modes 1 and 2 (AVX packets,
# fp64 accumulation) instead of 0, its J^T r moves by 0.8e-5 .. 3.1e-5 of sum|sd_k * pdiff| on these rows, against
# 0.2e-6 .. 0.8e-6 on the rows without dopatchnorm.
ROWS = [
    # ---- order 0, fast mode ----
    row("v8-8w-lvl1", FAST, "k_track_v8<false,false,8>", 2.2e-3, seed=401, psz=8, npts=100, ntracks=3, lv_l=1, **G8),
    row("v8-16w-motion", FAST, "k_track_v8<false,false,16>", 4.4e-3, edge=40, seed=402, psz=8, npts=200, ntracks=2,
        scale=3.0, **G8),
    row("v8-8w-pn", FAST, "k_track_v8<true,false,8>", 2.0e-3, jtr_tol=4.2e-5, seed=403, psz=8, npts=50, ntracks=3,
        dopatchnorm=1, **G8),
    row("v8-16w-pn-cap", FAST, "k_track_v8<true,false,16>", 7.2e-3, seed=404, psz=8, npts=260, maxpttrack=240,
        ntracks=2, dopatchnorm=1, **G8),
    row("v8-8w-donorm-pn", FAST, "k_track_v8<true,false,8>", 1.2e-2, jtr_tol=7.3e-5, p_in=P_START, seed=405, psz=8,
        npts=40, ntracks=3, donorm=1, dopatchnorm=1, **G8),
    row("fast8-250", FAST, "k_track_fast<8,4,4>", 8.6e-3, edge=60, seed=406, psz=8, npts=250, ntracks=2, **G8),
    row("fast16-9-donorm", FAST, "k_track_fast<16,4,4>", 5.1e-2, seed=407, psz=16, npts=9, ntracks=4, donorm=1, **G16),
    row("fast16-70", FAST, "k_track_fast<16,4,4>", 1.6e-2, seed=408, psz=16, npts=70, ntracks=2, **G16),
    row("fast32-18", FAST, "k_track_fast<32,16,4>", 7.2e-3, edge=6, seed=409, psz=32, npts=18, ntracks=2, **G32),
    row("v2-4-onept", FAST, "k_track_v2<16,4,false,256>", 1.4e-1, sizes=[4, 1, 4, 4], seed=410, psz=32, npts=4, **G32),
    row("v2-8", FAST, "k_track_v2<16,2,false,512>", 2.4e-2, edge=3, seed=411, psz=32, npts=8, ntracks=3, **G32),
    row("v2-16-lvl1", FAST, "k_track_v2<16,1,false,1024>", 1.5e-2, seed=412, psz=32, npts=16, ntracks=2, lv_l=1, **G32),
    row("general-psz4", FAST, "k_track<0,0>", 9.7e-4, edge=15, seed=413, psz=4, npts=50, ntracks=3, **G8),
    row("general-psz7-pn", FAST, "k_track<0,1>", 1.6e-3, jtr_tol=7.8e-5, seed=414, psz=7, npts=30, ntracks=3,
        dopatchnorm=1, **G8),
    row("general-psz16-pn", FAST, "k_track<16,1>", 7.4e-3, jtr_tol=4.6e-5, seed=415, psz=16, npts=40, ntracks=2,
        dopatchnorm=1, **G16),
    row("general-psz32-pn", FAST, "k_track<32,1>", 4.8e-2, jtr_tol=6.3e-5, seed=416, psz=32, npts=8, ntracks=2,
        dopatchnorm=1, **G32),
    row("multi-psz8-300", FAST, MULTI, 5.4e-3, seed=417, psz=8, npts=300, **G8),
    row("multi-psz8-242-pn", FAST, MULTI, 6.6e-3, edge=50, seed=418, psz=8, npts=242, dopatchnorm=1, **G8),
    row("multi-psz16-71", FAST, MULTI, 1.5e-2, seed=419, psz=16, npts=71, **G16),
    row("multi-psz32-19", FAST, MULTI, 7.8e-3, seed=420, psz=32, npts=19, **G32),
    row("dense-tma", FAST, DENSE_TMA, 1.4e-4, seed=421, psz=1, npts=3000, **G1),
    row("dense-ldg", FAST, DENSE_LDG, 2.1e-4, seed=422, psz=1, npts=3001, **G1),
    # ---- order 2, the general kernel forced ----
    row("o2-general-psz8", GENERAL, "k_track<8,0>", 3.5e-3, edge=20, seed=431, psz=8, npts=100, ntracks=3, **G8),
    row("o2-general-psz8-pn", GENERAL, "k_track<8,1>", 4.8e-3, seed=432, psz=8, npts=200, ntracks=2, dopatchnorm=1,
        **G8),
    row("o2-general-psz16", GENERAL, "k_track<16,0>", 8.1e-3, seed=433, psz=16, npts=70, ntracks=2, **G16),
    row("o2-general-psz32", GENERAL, "k_track<32,0>", 2.8e-2, seed=434, psz=32, npts=18, ntracks=2, **G32),
    row("o2-multi-psz1", GENERAL, MULTI, 1.9e-4, seed=435, psz=1, npts=3000, **G1),
    # ---- orders 1 and 3: the replay itself on real kernel output, bit for bit ----
    row("o1-k2r", SSE, "k_track_r<4,2>", seed=441, psz=32, npts=4, ntracks=4, **G32),
    row("o1-k2x8-donorm", SSE, "k_track_x8<false,15,1,4>", p_in=P_START, seed=442, psz=8, npts=100, ntracks=3, donorm=1,
        **G8),
    row("o3-k2x8", AVX, "k_track_x8<false,15,1,8>", edge=30, seed=443, psz=8, npts=100, ntracks=3, **G8),
    row("o1-multi-psz8", SSE, MULTI, seed=444, psz=8, npts=223, **G8),
]


def traced_name(want):
    """K2v8 and K2v2 take the trace as a template argument; the other kernels keep their names."""
    for head, pos in (("k_track_v8<", 1), ("k_track_v2<", 2)):
        if want.startswith(head):
            args = want[len(head):-1].split(",")
            args[pos] = "true"
            return head + ",".join(args) + ">"
    return want


def edge_points(sc, seed, n, k, psz, lv_f):
    """n points as synth.Scene.points places them, the first k moved to within 6 px of the left or right border."""
    rng = np.random.default_rng(4000 + seed)
    m = min(2 * psz * (1 << lv_f), sc.w // 4, sc.h // 4)
    u, v = rng.uniform(m, sc.w - m, n), rng.uniform(m, sc.h - m, n)
    left = rng.random(k) < 0.5
    u[:k] = np.where(left, rng.uniform(0.25, 6, k), sc.w - rng.uniform(0.25, 6, k))
    return sc.backproject(u, v)


def build_case(r):
    c = make_case(**r["kw"])
    if r["sizes"] is not None:
        psz, lv_f = c["psz"], c["lv_f"]
        c["pts"] = np.concatenate([c["sc"].points(500 + t, n, psz, lv_f) for t, n in enumerate(r["sizes"])])
        c["pt_off"] = np.concatenate([[0], np.cumsum(r["sizes"])]).astype(np.int64)
        c["T"] = len(r["sizes"])
    if r["edge"]:
        a = int(c["pt_off"][-2])
        n = int(c["pt_off"][-1]) - a
        c["pts"] = np.concatenate([c["pts"][:3 * a], edge_points(c["sc"], r["kw"]["seed"], n, r["edge"], c["psz"],
                                                                 c["lv_f"])])
    p_in = np.zeros((c["T"], 6)) if r["p_in"] is None else np.tile(np.asarray(r["p_in"], np.float64), (c["T"], 1))
    return c, p_in


def run_rows(ict, c, p_in, order, cap, profile=False):
    """The same tracking call untraced and traced; returns (untraced, traced, pyramids) or, with profile, the names of
    the kernels each of the two calls launched."""
    op = ict.OptParam.from_buffer_copy(bytes(c["op"]))
    fr = ict.Frames(2, c["w"], c["h"], c["lv_f"], c["psz"])
    tr = ict.Tracker(op, c["sc"].fc, c["sc"].cc, c["sc"].wh)
    try:
        fr.upload(0, np.stack([c["A"], c["B"]]))
        tr.set_sum_order(order)
        tr.set_points(c["pt_off"], c["pts"].copy())
        calls = (lambda: tr.track_batch(fr, 0, 1, p_in), lambda: tr.track_batch(fr, 0, 1, p_in, trace_cap=cap))
        if profile:
            return [kernels_of(f) for f in calls]
        return calls[0](), calls[1](), (fr.download(0), fr.download(1))
    finally:
        tr.close()
        fr.close()


def profile_rows(path):
    """Writes {row id: [untraced kernels, traced kernels]} for every row to path (JSON)."""
    import invcompcamtrack_b200 as ict
    ict.lib()
    out = {}
    for p in ROWS:
        r = p.values[0]
        c, p_in = build_case(r)
        out[p.id] = run_rows(ict, c, p_in, r["order"], replay_trace_cap(c["op"]), profile=True)
    with open(path, "w") as f:
        json.dump(out, f)


@pytest.fixture(scope="module")
def row_kernels(tmp_path_factory):
    """The kernels of every row, profiled in a fresh process.  Late in a long GPU session (after other tests have used
    torch's CUDA streams and pinned memory) the profiler has been seen to drop the record of a lone kernel launched on
    the default stream, while it still records the launch call; a fresh process profiles reliably."""
    path = str(tmp_path_factory.mktemp("replay") / "kernels.json")
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, HERE, os.environ.get("PYTHONPATH", "")]))
    r = subprocess.run([sys.executable, "-c", "import test_gpu_replay as m, sys; m.profile_rows(sys.argv[1])", path],
                       cwd=HERE, env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    with open(path) as f:
        return json.load(f)


@pytest.mark.gpu
@pytest.mark.parametrize("r", ROWS)
def test_replay(ict, orc, row_kernels, request, r):
    c, p_in = build_case(r)
    op, order = c["op"], r["order"]
    cap = replay_trace_cap(op)
    names0, names1 = row_kernels[request.node.callspec.id]
    assert_routed(names0, r["want"])
    assert_routed(names1, traced_name(r["want"]))
    g0, g, pyr = run_rows(ict, c, p_in, order, cap)

    check_trajectory(g, op)
    orc.set_sum_mode(ORACLE_MODE[order])
    try:
        rep = replay_batch(replay_models(orc, c, pyr, p_in), g["trace"])
    finally:
        orc.set_sum_mode(0)
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
        jtr, dp, nrec = teacher_forced_errors(g, dict(trace=m))
        msg = "J^T r %.2e of sum|sd*r|, delta_p %.2e of the level's first step" % (jtr, dp)
        assert jtr <= r["jtr_tol"], msg
        assert dp <= r["dp_tol"], msg
    nrec = int((g["trace"][..., 0] >= 0).sum())
    print("replay %s: %s, %d records, %d nvis flips at the bounds, levels %s" % (
        names1[0] if len(set(names1)) == 1 else r["want"], msg, nrec, nflip, g["iters"].tolist()))
    for k in ("p_out", "iters", "npixres"):
        assert np.array_equal(g0[k], g[k]), k
