"""Sum order 3 (ict_tracker_set_sum_order): the reference's order of summation with Eigen's 8-float AVX packets —
sixteen sequential chains per sum, then predux(lo + hi) — against the oracle in its sum mode 1, BIT FOR BIT: every
iteration's J^T r and delta_p, iteration counts, pixel-residual counts and final poses, through every kernel that
takes the order (the general kernel, K2x8 at psz 8 and 16 in both launch forms, the multi-CTA path) and every tracking
entry point."""
import numpy as np
import pytest

from helpers import make_case, oracle_run, gpu_run, assert_bit_identical

AVX = 3          # ict_tracker_set_sum_order
ORACLE_AVX = 1   # ict_oracle_set_sum_mode

# the single-track cases of tests/test_gpu_parity.py
CASES = [
    dict(seed=0),                                            # BASELINE config 1: 640x480, psz 8, 100 points
    dict(seed=1, donorm=1),
    dict(seed=2, dopatchnorm=1),
    dict(seed=3, donorm=1, dopatchnorm=1),
    dict(seed=4, psz=4, npts=50),
    dict(seed=5, psz=16, npts=17),
    dict(seed=6, psz=7, npts=20),                            # odd psz: shifted placement (SURVEY §9.3)
    dict(seed=7, psz=32, npts=4, w=1920, h=1080),            # config 3 geometry, one track
    dict(seed=8, lv_f=2, lv_l=1, maxiter=5, ratio=0.1),
    dict(seed=9, npts=37, maxpttrack=24),                    # more points than maxpttrack: the rest is ignored
    dict(seed=10, scale=3.0),                                # large motion: points leave the new frame at some levels
]


def check(ict, orc, case, trace_cap=64, p_in=None, pyramids=False):
    o = oracle_run(orc, case, trace_cap=trace_cap, sum_mode=ORACLE_AVX, p_in=p_in)
    g = gpu_run(ict, case, trace_cap=trace_cap, sum_order=AVX, p_in=p_in)
    if pyramids:
        for k in range(3):
            assert np.array_equal(g["pyr"][0][k], o["pyr"][0][k])
            assert np.array_equal(g["pyr"][1][k], o["pyr"][1][k])
    assert np.array_equal(g["pt2d"], o["pt2d"])              # reference reprojection (2-D points)
    assert_bit_identical(g, o)
    return g, o


def test_cases_tell_the_orders_apart(orc):
    """The oracle's two packet orders give different per-iteration traces on every case below, so bit-identity with
    mode 1 says something that bit-identity with mode 0 does not."""
    for kw in CASES:
        case = make_case(**kw)
        o0 = oracle_run(orc, case, sum_mode=0)
        o1 = oracle_run(orc, case, sum_mode=ORACLE_AVX)
        assert not np.array_equal(o0["trace"][..., 2:8], o1["trace"][..., 2:8]), kw


@pytest.mark.gpu
@pytest.mark.parametrize("kw", CASES, ids=[str(i) for i in range(len(CASES))])
def test_track_bit_exact_in_avx_order(ict, orc, kw):
    check(ict, orc, make_case(**kw), pyramids=True)


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(seed=31, ntracks=64),                                     # C1 x 64
                                dict(seed=21, w=1920, h=1080, psz=32, npts=4, ntracks=256)],   # psz 32: general kernel
                         ids=["c1x64", "psz32x256"])
def test_batches(ict, orc, kw):
    check(ict, orc, make_case(**kw), trace_cap=48)


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(npts=24, ntracks=170), dict(npts=24, ntracks=170, dopatchnorm=1, donorm=1)])
def test_psz8_both_launch_forms(ict, orc, kw):
    """K2x8 with seven producer warps (170 tracks > SM count) and with fifteen (a 9-track sub-batch): bit-identical to
    the oracle, and a track's result independent of the form its batch took."""
    case = make_case(seed=311, psz=8, **kw)
    g, _ = check(ict, orc, case, trace_cap=48)
    sub = dict(case, T=9, pt_off=case["pt_off"][:10], pts=case["pts"][:3 * int(case["pt_off"][9])])
    gs, _ = check(ict, orc, sub, trace_cap=48)
    assert np.array_equal(gs["p_out"], g["p_out"][:9]) and np.array_equal(gs["iters"], g["iters"][:9])


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(psz=8, npts=150, ntracks=2), dict(psz=8, npts=224, ntracks=2),
                                dict(psz=8, npts=200, dopatchnorm=1, ntracks=2),
                                dict(psz=16, npts=9, ntracks=5, w=960, h=544), dict(psz=16, npts=20, ntracks=170, w=960, h=544),
                                dict(psz=16, npts=30, scale=3.0, ntracks=8, w=960, h=544)],
                         ids=["psz8-150", "psz8-224", "psz8-200-pn", "psz16-9", "psz16-20x170", "psz16-30-large"])
def test_k2x8(ict, orc, kw):
    check(ict, orc, make_case(seed=321, **kw), trace_cap=48)


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(seed=80, psz=8, npts=230),                                 # beyond one CTA
                                dict(seed=81, psz=8, npts=240, donorm=1, dopatchnorm=1),
                                dict(seed=61, w=320, h=240, lv_f=2, psz=1, dense_border=8, tilt=(0.15, -0.1)),
                                dict(seed=62, w=320, h=240, lv_f=2, psz=1, dense_border=6, tilt=(0.1, 0.2), donorm=1),
                                dict(seed=63, w=160, h=120, lv_f=1, psz=8, npts=900),
                                dict(seed=64, w=160, h=120, lv_f=1, psz=8, npts=700, donorm=1, dopatchnorm=1),
                                dict(seed=65, w=640, h=480, psz=8, npts=4200)],
                         ids=["psz8-230", "psz8-240-pn", "dense", "dense-donorm", "psz8-900", "psz8-700-pn", "psz8-4200"])
def test_multi_cta_path(ict, orc, kw):
    """Tracks too large for one CTA (dense psz 1 among them): the multi-CTA path with sixteen chains per sum, in its
    three-launch (no dopatchnorm, up to 2^18 pixel slots) and five-launch (dopatchnorm, or more slots) iteration forms."""
    case = make_case(**kw)
    check(ict, orc, case, trace_cap=48)


@pytest.mark.gpu
def test_several_large_tracks_per_call(ict, orc):
    check(ict, orc, make_case(psz=8, seed=85, npts=600, ntracks=3, w=640, h=480), trace_cap=48)


@pytest.mark.gpu
def test_sequence_chain(ict, orc):
    """A forward chain over 6 frames (ict_track_sequence) against the oracle's chain, pose by pose."""
    from invcompcamtrack_b200 import synth
    from oracle import oracle as O
    nfr = 6
    sc, frames, poses = synth.make_sequence(3, nfr, 320, 240)
    op_o = O.make_optparam(lv_f=2, psz=8, maxpttrack=60)
    pts = sc.points(77, 60, 8, 2)
    pyr = [orc.pyramid_build(f.astype(np.float32), 2, 8) for f in frames]
    p = np.zeros((1, 6))
    chain, iters = [p.copy()], []
    orc.set_sum_mode(ORACLE_AVX)
    try:
        for k in range(nfr - 1):
            r = orc.track_batch(op_o, sc.fc, sc.cc, sc.wh, [q[0] for q in pyr], [q[1] for q in pyr], [q[2] for q in pyr],
                                np.array([0, 60]), pts.copy(), [k], [k + 1], p)
            p = r["p_out"]
            chain.append(p.copy())
            iters.append(r["iters"])
    finally:
        orc.set_sum_mode(0)
    op = ict.OptParam.from_buffer_copy(bytes(op_o))
    fr = ict.Frames(nfr, 320, 240, 2, 8)
    fr.upload(0, np.stack(frames))
    tr = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
    tr.set_points(np.array([0, 60]), pts.copy())
    tr.set_sum_order(AVX)
    g = tr.track_sequence(fr, 0, nfr - 1, 1, np.zeros(6))
    for k in range(nfr):
        assert np.array_equal(g["poses"][k, 0], chain[k][0]), k
    for k in range(nfr - 1):
        assert np.array_equal(g["iters"][k], iters[k]), k
    tr.close(); fr.close()


@pytest.mark.gpu
def test_keep_state_across_calls(ict, orc):
    """keep_state in order 3: after ONE set_points, several track_batch calls on a pan in which points leave the frame
    (they keep the template of the last level they were visible at, possibly from an earlier call).  The oracle's
    OdometerClass does the same when driven through the same SetPose / TrackPose calls after a single Set3Dpoints: it
    resets its arrays only there."""
    from invcompcamtrack_b200 import synth
    from oracle import oracle as O
    w, h, nb, nf = 160, 120, 2, 3                  # the geometry of run_track_nposes with points leaving the frames
    sc = synth.Scene(19, w, h)
    nfr = nb + nf + 1
    poses = np.zeros((nfr, 6))
    for k in range(nfr):
        poses[k] = np.array([0.22 * (k - nb), 0.02 * (k - nb), 0.0, 0.0, 0.0, 0.004 * (k - nb)])
    frames = [sc.render(poses[k]) for k in range(nfr)]
    rng = np.random.default_rng(14)
    n = 64
    u = np.concatenate([rng.uniform(1, 12, n // 4), rng.uniform(w - 12, w - 1, n // 4), rng.uniform(20, w - 20, n // 2)])
    v = rng.uniform(10, h - 10, n)
    pts = sc.backproject(u, v, poses[nb])
    lv_f = 2
    steps = [(nb, nb + 1), (nb + 1, nb + 2), (nb + 2, nb + 3), (nb + 3, nb + 2), (nb, nb - 1), (nb - 1, nb - 2)]

    op_o = O.make_optparam(lv_f=lv_f, psz=8, maxiter=10, normdp_ratio=0.01, maxpttrack=n)
    pyr = [orc.pyramid_build(f.astype(np.float32), lv_f, 8) for f in frames]
    _, offs, _, _ = O.pyramid_layout(w, h, lv_f, 8)
    od = O.Odometer(orc, op_o, sc.fc, sc.cc, sc.wh)
    want = []
    orc.set_sum_mode(ORACLE_AVX)
    try:
        od.set3dpoints(pts.copy())
        for a, b in steps:
            od.setpose(poses[a], pyr[a], pyr[b], lv_f, offs)
            p = od.trackpose()
            it = np.ctypeslib.as_array(orc.lib.ict_oracle_last_iters(od.h), shape=(lv_f + 1,)).copy()
            want.append((p, it, int(orc.lib.ict_oracle_last_npixres(od.h))))
    finally:
        orc.set_sum_mode(0)
        od.close()

    op = ict.OptParam.from_buffer_copy(bytes(op_o))
    fr = ict.Frames(nfr, w, h, lv_f, 8)
    fr.upload(0, np.stack(frames))
    tr = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
    tr.set_sum_order(AVX)
    tr.set_knob("keep_state", 1)
    tr.set_points(np.array([0, n]), pts.copy())
    fresh = ict.Tracker(op, sc.fc, sc.cc, sc.wh)       # without the carried state, for contrast
    fresh.set_sum_order(AVX)
    fresh.set_points(np.array([0, n]), pts.copy())
    differs = False
    for (a, b), (p, it, npx) in zip(steps, want):
        g = tr.track_batch(fr, a, b, poses[a][None])
        assert np.array_equal(g["p_out"][0], p), (a, b)
        assert np.array_equal(g["iters"][0], it) and int(g["npixres"][0]) == npx, (a, b)
        differs |= not np.array_equal(fresh.track_batch(fr, a, b, poses[a][None])["p_out"][0], p)
    assert differs, "the pan must make the carried state matter"
    tr.close(); fresh.close(); fr.close()


@pytest.mark.gpu
def test_switching_orders_and_bad_order(ict, orc):
    """set_sum_order(3) then (1) is order 1 bit for bit; 4 and -1 are refused with ICT_ERR_BAD_ARG."""
    from invcompcamtrack_b200.api import IctError
    case = make_case(seed=5, psz=16, npts=17)
    o = oracle_run(orc, case, sum_mode=0)
    op = ict.OptParam.from_buffer_copy(bytes(case["op"]))
    fr = ict.Frames(2, case["w"], case["h"], case["lv_f"], case["psz"])
    fr.upload(0, np.stack([case["A"], case["B"]]))
    tr = ict.Tracker(op, case["sc"].fc, case["sc"].cc, case["sc"].wh)
    tr.set_points(case["pt_off"], case["pts"].copy())
    tr.set_sum_order(AVX)
    a = tr.track_batch(fr, 0, 1, np.zeros((1, 6)), trace_cap=64)
    tr.set_sum_order(1)
    b = tr.track_batch(fr, 0, 1, np.zeros((1, 6)), trace_cap=64)
    assert_bit_identical(b, o)
    assert not np.array_equal(a["trace"][..., 2:8], b["trace"][..., 2:8])
    for bad in (4, -1):
        with pytest.raises(IctError, match="ICT_ERR_BAD_ARG"):
            tr.set_sum_order(bad)
    tr.close(); fr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(psz=8, npts=100, ntracks=300), dict(psz=16, npts=9, ntracks=40, w=960, h=544),
                                dict(psz=32, npts=4, ntracks=200, w=1280, h=704)], ids=["psz8", "psz16", "psz32"])
def test_stream_entry_points_equal_blocking_ones(ict, kw):
    """ict_tracker_set_points_stream + ict_track_batch_stream in order 3 give the blocking call's results."""
    import ctypes as C
    import torch
    case = make_case(seed=95, **kw)
    T, P, L = case["T"], case["npts"], case["lv_f"] + 1
    op = ict.OptParam.from_buffer_copy(bytes(case["op"]))
    fr = ict.Frames(2, case["w"], case["h"], case["lv_f"], case["psz"])
    fr.upload(0, np.stack([case["A"], case["B"]]))
    tr = ict.Tracker(op, case["sc"].fc, case["sc"].cc, case["sc"].wh)
    tr.set_sum_order(AVX)
    tr.set_points(case["pt_off"], case["pts"].copy())
    ref = tr.track_batch(fr, 0, 1, np.zeros((T, 6)))
    tr.close()
    lib, v = ict.lib(), C.c_void_p
    st = torch.cuda.Stream()
    h_off = torch.from_numpy(case["pt_off"].copy()).pin_memory()
    h_pts = torch.from_numpy(case["pts"].copy()).pin_memory()
    h_ref = torch.zeros(T, dtype=torch.int32).pin_memory()
    h_new = torch.ones(T, dtype=torch.int32).pin_memory()
    h_pin = torch.zeros(T, 6, dtype=torch.float64).pin_memory()
    h_pout = torch.zeros(T, 6, dtype=torch.float64).pin_memory()
    h_iters = torch.zeros(T, L, dtype=torch.int32).pin_memory()
    h_npix = torch.zeros(T, dtype=torch.int64).pin_memory()
    ts = ict.Tracker(op, case["sc"].fc, case["sc"].cc, case["sc"].wh)
    ts.set_sum_order(AVX)
    for step in range(2):
        h_pout.zero_()
        rc = lib.ict_tracker_set_points_stream(ts.h_, T, v(h_off.data_ptr()), v(h_pts.data_ptr()), v(st.cuda_stream))
        rc |= lib.ict_track_batch_stream(ts.h_, fr.h_, v(h_ref.data_ptr()), v(h_new.data_ptr()), v(h_pin.data_ptr()),
                                         v(h_pout.data_ptr()), v(h_iters.data_ptr()), v(h_npix.data_ptr()),
                                         v(st.cuda_stream))
        assert rc == 0, lib.ict_last_error()
        st.synchronize()
        assert np.array_equal(h_pout.numpy(), ref["p_out"]), step
        assert np.array_equal(h_iters.numpy(), ref["iters"]) and np.array_equal(h_npix.numpy(), ref["npixres"])
    ts.close(); fr.close()


EXTREME = [
    dict(psz=32, w=1280, h=704, npts=4, ntracks=10),     # general kernel
    dict(psz=8, npts=60, ntracks=10),                    # K2x8
    dict(psz=16, npts=9, ntracks=10),                    # K2x8, four tiles per patch
]


@pytest.mark.gpu
@pytest.mark.parametrize("kw", EXTREME, ids=["psz32", "psz8", "psz16"])
def test_extreme_poses_stay_in_bounds(ict, orc, kw):
    """Poses that throw the patch centres far outside the padded planes, behind the camera or to infinity: order 3 is
    bit-identical to the oracle (an out-of-bounds read would have to return the oracle's values) and deterministic;
    non-finite initial poses place no patch at all; an ordinary run afterwards is still bit-identical."""
    case = make_case(seed=301, **kw)
    T = case["T"]
    p_in = np.zeros((T, 6))
    p_in[0, 0] = 1e6
    p_in[1, 1] = -3e4
    p_in[2, 2] = -50.0
    p_in[3, 2] = -1.0
    p_in[4, 3] = np.pi
    p_in[5, 4] = 0.5 * np.pi
    p_in[6, 5] = 3.0
    p_in[7, :3] = (1e20, -1e20, 1e20)
    p_in[8, 2] = 1e6
    p_in[9, :] = (0.3, -0.2, 0.1, 0.2, -0.3, 0.1)
    g, _ = check(ict, orc, case, trace_cap=48, p_in=p_in)
    gb = gpu_run(ict, case, trace_cap=48, sum_order=AVX, p_in=p_in)
    assert np.array_equal(g["p_out"], gb["p_out"], equal_nan=True) and np.array_equal(g["iters"], gb["iters"])
    p_bad = np.zeros((T, 6))
    p_bad[0, 0] = np.nan
    p_bad[1, 4] = np.inf
    gn = gpu_run(ict, case, trace_cap=0, sum_order=AVX, p_in=p_bad)
    assert gn["npixres"][0] == 0 and gn["npixres"][1] == 0
    assert np.isfinite(gn["p_out"][2:]).all()
    check(ict, orc, case, trace_cap=48)
