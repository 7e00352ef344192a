"""GPU parity tests: the CUDA path through the C ABI vs the CPU oracle on identical seeded inputs."""
import numpy as np
import pytest

from helpers import (make_case, oracle_run, gpu_run, check_parity, assert_bit_identical,
                     check_against_oracle_spread)

pytestmark = pytest.mark.gpu


def test_device_present(ict):
    assert ict.device_count() >= 1


@pytest.mark.parametrize("w,h,lv_f,pad", [(640, 480, 3, 8), (160, 120, 1, 8), (320, 240, 2, 5), (1920, 1080, 3, 32),
                                           (64, 48, 3, 1)])
def test_pyramid_bit_exact(ict, orc, w, h, lv_f, pad):
    rng = np.random.default_rng(w + lv_f)
    img = rng.integers(0, 256, (h, w)).astype(np.float32)
    g = ict.pyramid_build(img, lv_f, pad)
    o = orc.pyramid_build(img, lv_f, pad)
    for k in range(3):
        assert np.array_equal(g[k], o[k])


def test_pyramid_u8_upload_equals_float(ict):
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (2, 96, 128)).astype(np.uint8)
    fa = ict.Frames(2, 128, 96, 2, 8); fa.upload(0, img)
    fb = ict.Frames(2, 128, 96, 2, 8); fb.upload(0, img.astype(np.float32))
    for f in range(2):
        for a, b in zip(fa.download(f), fb.download(f)):
            assert np.array_equal(a, b)


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


@pytest.mark.parametrize("kw", CASES, ids=[str(i) for i in range(len(CASES))])
def test_track_bit_exact_in_reference_order(ict, orc, kw):
    """With the reductions run in the reference's order the CUDA path reproduces the oracle BIT FOR BIT: pyramids,
    reference reprojection, every iteration's J^T r and delta_p, iteration counts, final pose."""
    case = make_case(**kw)
    o = oracle_run(orc, case)
    g = gpu_run(ict, case, sum_order=1)
    for k in range(3):
        assert np.array_equal(g["pyr"][0][k], o["pyr"][0][k])
        assert np.array_equal(g["pyr"][1][k], o["pyr"][1][k])
    assert np.array_equal(g["pt2d"], o["pt2d"])              # reference reprojection
    assert_bit_identical(g, o)


@pytest.mark.parametrize("kw", CASES, ids=[str(i) for i in range(len(CASES))])
def test_track_parity_fast_order(ict, orc, kw):
    """Default (tree) reductions on identical inputs: first-iteration J^T r within 1e-5 relative of the oracle.  A
    single track cannot carry statistical gates; the batches below do."""
    case = make_case(**kw)
    o = oracle_run(orc, case)
    g = gpu_run(ict, case)
    assert np.array_equal(g["pt2d"], o["pt2d"])
    res = check_parity(g, o, case, gates=False)
    assert res["jtr_first"] <= 1e-5, res
    assert np.abs(g["p_out"][0] - o["p_out"][0]).max() < 5e-3, res      # same basin, same answer up to noise
    print(kw, res, g["iters"][0])


def test_track_bit_exact_batch(ict, orc):
    """256 independent tracks of 4 points, 32x32 patches, 1080p (BASELINE config 3 geometry, reduced count)."""
    case = make_case(seed=21, w=1920, h=1080, psz=32, npts=4, ntracks=256)
    o = oracle_run(orc, case, trace_cap=48)
    g = gpu_run(ict, case, trace_cap=48, sum_order=1)
    assert np.array_equal(g["pt2d"], o["pt2d"])
    assert_bit_identical(g, o)


def test_track_parity_batch_fast_order(ict, orc):
    """Same batch with the default tree reductions.  4-point tracks are ill-conditioned: the reference itself moves
    by ~1e-2 relative in translation and flips ~13 % of its stopping decisions when only its summation order changes
    (oracle modes), so the gate is the oracle's own spread, not an absolute 1e-5."""
    case = make_case(seed=21, w=1920, h=1080, psz=32, npts=4, ntracks=256)
    g = gpu_run(ict, case, trace_cap=48)
    m, spread = check_against_oracle_spread(g, case, orc, trace_cap=48)
    print("gpu", m, "oracle spread", spread)


def test_track_parity_c1_many(ict, orc):
    """BASELINE config 1 geometry (640x480, psz 8, 100 points) x 64 tracks: bit-exact in reference order; in the
    default order within the oracle's own spread AND close to the north_star numbers (well-conditioned problem)."""
    case = make_case(seed=31, ntracks=64)
    o = oracle_run(orc, case)
    gx = gpu_run(ict, case, sum_order=1)
    assert_bit_identical(gx, o)
    g = gpu_run(ict, case)
    m, spread = check_against_oracle_spread(g, case, orc)
    assert m["frac_same"] >= 0.95 and m["worst_rot"] <= 1e-5 and m["median_tr"] <= 1e-5 and m["worst_tr"] <= 1e-4, m
    print("gpu", m, "oracle spread", spread)


@pytest.mark.parametrize("kw", [dict(seed=51, ntracks=8), dict(seed=52, psz=16, npts=9, ntracks=5),
                                dict(seed=53, psz=32, npts=4, w=1920, h=1080, ntracks=64),
                                dict(seed=54, psz=32, npts=7, w=1920, h=1080, ntracks=3), dict(seed=55, scale=3.0, ntracks=4),
                                dict(seed=56, npts=37, maxpttrack=24, ntracks=3), dict(seed=57, donorm=1, ntracks=4)])
def test_fast_kernel_equals_general_kernel_up_to_sum_order(ict, orc, kw):
    """k_track_fast (production) and k_track (general) run the same per-pixel arithmetic; only the order of the tree
    sums differs.  First-iteration J^T r must agree to fp32 summation noise, both with the oracle and each other,
    and both must count the same pixel-residuals on the first iterations."""
    case = make_case(**kw)
    o = oracle_run(orc, case)
    gf = gpu_run(ict, case, sum_order=0)
    gg = gpu_run(ict, case, sum_order=2)
    assert np.array_equal(gf["pt2d"], gg["pt2d"]) and np.array_equal(gf["pt2d"], o["pt2d"])
    for g in (gf, gg):
        res = check_parity(g, o, case, gates=False)
        assert res["jtr_first"] <= 1e-5, res
        assert np.array_equal(g["trace"][:, 0, 15], o["trace"][:, 0, 15])      # visible points, first iteration
    assert np.abs(gf["p_out"] - gg["p_out"]).max() < 5e-3


def test_track_pair_entry_point(ict, orc):
    case = make_case(seed=41, donorm=1)
    o = oracle_run(orc, case)
    op = ict.OptParam.from_buffer_copy(bytes(case["op"]))
    pts = case["pts"].copy()
    r = ict.track_pair(op, case["sc"].fc, case["sc"].cc, case["sc"].wh, case["A"], case["B"], pts, np.zeros(6),
                       trace_cap=64)
    g = dict(p_out=r["p_out"][None], iters=r["iters"][None], trace=r["trace"][None])
    # one track in the default order: identical inputs -> J^T r to summation noise; afterwards the trajectory may
    # separate from the oracle's like the oracle's own summation orders do (statistics: profiles/tools/
    # solve_agreement.py, test_track_parity_c1_many), but it ends at the same pose
    res = check_parity(g, o, case, gates=False)
    assert res["jtr_first"] <= 1e-5, res
    assert np.abs(g["p_out"][0] - o["p_out"][0]).max() < 1e-4, (g["p_out"], o["p_out"])
    # donorm: the caller's points were centred in place, like odometer.cpp:207-212
    assert abs(pts[:case["npts"]].mean()) < 1e-9 and not np.allclose(pts, case["pts"])


def test_sequence_chain(ict, orc):
    """Forward chain over 6 frames == run_track_nposes.cpp:232-239; GPU chain vs oracle chain, pose by pose."""
    from invcompcamtrack_b200 import synth
    from oracle import oracle as O
    nfr = 6
    sc, frames, poses = synth.make_sequence(3, nfr, 320, 240)
    op_o = O.make_optparam(lv_f=2, psz=8, maxpttrack=60)
    pts = sc.points(77, 60, 8, 2)
    pyr = [orc.pyramid_build(f.astype(np.float32), 2, 8) for f in frames]
    p = np.zeros((1, 6))
    chain = [p.copy()]
    for k in range(nfr - 1):
        r = orc.track_batch(op_o, sc.fc, sc.cc, sc.wh, [q[0] for q in pyr], [q[1] for q in pyr], [q[2] for q in pyr],
                            np.array([0, 60]), pts.copy(), [k], [k + 1], p)
        p = r["p_out"]
        chain.append(p.copy())
    op = ict.OptParam.from_buffer_copy(bytes(op_o))
    fr = ict.Frames(nfr, 320, 240, 2, 8)
    fr.upload(0, np.stack(frames))
    tr = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
    tr.set_points(np.array([0, 60]), pts.copy())
    tr.set_sum_order(1)                                   # reference order: the whole chain is bit-identical
    g = tr.track_sequence(fr, 0, nfr - 1, 1, np.zeros(6))
    for k in range(nfr):
        assert np.array_equal(g["poses"][k, 0], chain[k][0]), k
    tr.set_sum_order(0)                                   # default order: same chain up to fp32 summation noise
    g = tr.track_sequence(fr, 0, nfr - 1, 1, np.zeros(6))
    for k in range(nfr):
        assert np.abs(g["poses"][k, 0] - chain[k][0]).max() < 1e-4, k
    # and the chain actually follows the ground-truth motion
    assert np.abs(g["poses"][-1, 0] - poses[-1]).max() < 2e-2
    # backward chain from the last frame returns to the start (run_track_nposes.cpp:251-258)
    b = tr.track_sequence(fr, nfr - 1, nfr - 1, -1, g["poses"][-1, 0])
    assert np.abs(b["poses"][-1, 0]).max() < 2e-2


@pytest.mark.parametrize("kw", [dict(npts=60, S=7), dict(npts=150, S=3, donorm=1, dopatchnorm=1)])
def test_chain_in_one_launch_equals_per_frame_launches(ict, kw):
    """ict_track_sequence with psz 8 in the fast mode: K2v8 loops over the frames inside ONE launch (a track's step
    k+1 depends on its own step k only).  Same poses, iteration counts and pixel-residual counts, bit for bit, as one
    launch per frame (tracker knob "seq_launches"), forwards and backwards."""
    from invcompcamtrack_b200 import synth
    nfr, S, n = 6, kw["S"], kw["npts"]
    sc, frames, poses = synth.make_sequence(3, nfr, 320, 240)
    op = ict.make_optparam(lv_f=2, psz=8, maxpttrack=n, donorm=kw.get("donorm", 0), dopatchnorm=kw.get("dopatchnorm", 0))
    fr = ict.Frames(nfr, 320, 240, 2, 8)
    fr.upload(0, np.stack(frames))
    tr = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
    tr.set_sum_order(0)                              # the chain-in-one-launch kernel is the fast mode's K2v8
    tr.set_points(np.arange(S + 1, dtype=np.int64) * n, np.concatenate([sc.points(70 + s, n, 8, 2) for s in range(S)]))
    p0 = np.zeros((S, 6))
    p0[:, 3] = np.linspace(-0.01, 0.01, S)          # chains that start apart
    a = tr.track_sequence(fr, 0, nfr - 1, 1, p0)
    ab = tr.track_sequence(fr, nfr - 1, nfr - 1, -1, a["poses"][-1])
    tr.set_knob("seq_launches", 1)
    b = tr.track_sequence(fr, 0, nfr - 1, 1, p0)
    bb = tr.track_sequence(fr, nfr - 1, nfr - 1, -1, b["poses"][-1])
    for x, y in ((a, b), (ab, bb)):
        assert np.array_equal(x["poses"], y["poses"])
        assert np.array_equal(x["iters"], y["iters"]) and np.array_equal(x["npixres"], y["npixres"])
    if not kw.get("donorm"):                                          # and the chains follow the motion
        assert np.abs(a["poses"][-1] - poses[-1]).max() < 5e-2
    tr.close(); fr.close()


@pytest.mark.parametrize("kw", [dict(seed=61, w=320, h=240, lv_f=2, psz=1, dense_border=8, tilt=(0.15, -0.1)),
                                dict(seed=62, w=320, h=240, lv_f=2, psz=1, dense_border=6, tilt=(0.1, 0.2), donorm=1),
                                dict(seed=63, w=160, h=120, lv_f=1, psz=8, npts=900),
                                dict(seed=64, w=160, h=120, lv_f=1, psz=8, npts=700, donorm=1, dopatchnorm=1),
                                dict(seed=65, w=640, h=480, psz=8, npts=4200)])   # 268 800 slots: streaming ref. order
def test_dense_alignment_multi_cta_path(ict, orc, kw):
    """BASELINE config 4 geometry (reduced): one track with one point per pixel and per-pixel depth, psz = 1 — too
    large for a CTA, so the multi-CTA path runs.  Bit-exact against the oracle in reference order; within fp32
    summation noise in the default order; recovers the ground-truth motion."""
    case = make_case(**kw)
    assert case["npts"] * case["op"].novals * 12 > 227 * 1024
    o = oracle_run(orc, case, trace_cap=48)
    gx = gpu_run(ict, case, trace_cap=48, sum_order=1)
    assert np.array_equal(gx["pt2d"], o["pt2d"])
    assert_bit_identical(gx, o)
    g = gpu_run(ict, case, trace_cap=48)
    res = check_parity(g, o, case, gates=False)
    assert res["jtr_first"] <= 1e-5, res
    assert np.abs(g["p_out"][0] - o["p_out"][0]).max() < 1e-3, res
    if kw["psz"] == 1:   # psz = 1 samples both images one pixel up-left (SURVEY §9.3): biased but it follows the motion
        assert np.abs(g["p_out"][0] - case["p_gt"]).max() < 0.25 * np.abs(case["p_gt"]).max()
        # the fused dense kernels (one launch per iteration) against the general multi-CTA kernels in the same tree
        # order: same per-element arithmetic, same partition, same summation order -> equal bits
        gg = gpu_run(ict, case, trace_cap=48, sum_order=2)
        assert np.array_equal(g["p_out"], gg["p_out"]) and np.array_equal(g["iters"], gg["iters"])
        assert np.array_equal(g["npixres"], gg["npixres"])
        assert np.array_equal(g["trace"][..., :16], gg["trace"][..., :16])
    print(res, g["iters"], o["iters"])


def test_several_large_tracks_per_call(ict, orc):
    """Tracks beyond one CTA (300 points of 8x8 pixels) in one ict_track_batch call: the multi-CTA path takes them one
    after the other on the stream.  Reference order: bit-identical to the oracle, track by track."""
    case = make_case(psz=8, seed=85, npts=300, ntracks=3, w=640, h=480)
    o = oracle_run(orc, case, trace_cap=48)
    gx = gpu_run(ict, case, trace_cap=48, sum_order=1)
    assert np.array_equal(gx["pt2d"], o["pt2d"])
    assert_bit_identical(gx, o)
    g = gpu_run(ict, case, trace_cap=48)
    res = check_parity(g, o, case, gates=False)
    assert res["jtr_first"] <= 1e-5, res
    assert np.abs(g["p_out"] - o["p_out"]).max() < 1e-3, res


@pytest.mark.parametrize("psz,patchnorm", [(8, 0), (8, 1), (7, 1), (32, 0), (4, 1)])
def test_get_patches_equal_the_oracle(ict, orc, psz, patchnorm):
    """ict_get_patches == util_getPatch / util_getPatch_grad (utilities.cpp:55-189), bit for bit, including the
    ceil(x + 1e-5f) placement at integer coordinates below and above 256, odd patch sizes and the patch mean in Eigen's
    summation order."""
    from invcompcamtrack_b200 import synth
    from oracle import oracle as O
    sc, A, B, _ = synth.make_pair(31, 640, 480)
    lv_f = 2
    fr = ict.Frames(1, 640, 480, lv_f, psz)
    fr.upload(0, A[None].astype(np.float32))
    pyr = orc.pyramid_build(A.astype(np.float32), lv_f, psz)
    _, off, sw, sh = O.pyramid_layout(640, 480, lv_f, psz)
    op = ict.make_optparam(lv_f=lv_f, psz=psz, dopatchnorm=patchnorm, maxpttrack=4)
    op_o = O.make_optparam(lv_f=lv_f, psz=psz, dopatchnorm=patchnorm, maxpttrack=4)
    rng = np.random.default_rng(5)
    for lvl in range(lv_f + 1):
        wl, hl = 640 >> lvl, 480 >> lvl
        mids = np.concatenate([rng.uniform([0, 0], [wl, hl], (24, 2)),
                               [[5.0, 7.0], [255.0, 100.0], [256.0, 30.0], [300.0, 17.0], [0.0, 0.0], [wl, hl],
                                [12.999995, 40.5]]]).astype(np.float32)
        mids = mids[(mids[:, 0] <= wl) & (mids[:, 1] <= hl)]
        I, dx, dy = fr.get_patches(0, lvl, op, mids)
        n = sw[lvl] * sh[lvl]
        planes = [pyr[k][off[lvl]:off[lvl] + n] for k in range(3)]
        for i, m in enumerate(mids):
            ref = orc.getpatch_grad(planes[0], planes[1], planes[2], m, op_o, sw[lvl])
            assert np.array_equal(I[i], ref[0]) and np.array_equal(dx[i], ref[1]) and np.array_equal(dy[i], ref[2]), (lvl, m)
        only = fr.get_patches(0, lvl, op, mids, grad=False)
        for i, m in enumerate(mids[:6]):
            assert np.array_equal(only[i], orc.getpatch(planes[0], m, op_o, sw[lvl]))
    fr.close()


def test_ncc_scoring(ict, orc):
    """run_track_nposes.cpp:271-355 on the GPU vs the oracle: per-point weighted NCC of back / reference / forward
    patches, including points outside the frames (corr = -1 when the reference point is out, weight 0 otherwise)."""
    from invcompcamtrack_b200 import synth
    from oracle import oracle as O
    sc, frames, poses = synth.make_sequence(5, 3, 320, 240)
    op_o = O.make_optparam(lv_f=2, psz=8, maxpttrack=64)
    rng = np.random.default_rng(3)
    n = 64
    def pts2d(jit):
        x = rng.uniform(-5, 325, n).astype(np.float32); y = rng.uniform(-5, 245, n).astype(np.float32)
        return np.concatenate([x, y])
    pr = pts2d(0)
    pb = (pr + rng.normal(0, 0.7, 2 * n)).astype(np.float32)
    pf = (pr + rng.normal(0, 0.7, 2 * n)).astype(np.float32)
    pyr = [orc.pyramid_build(f.astype(np.float32), 2, 8) for f in frames]
    ref = orc.ncc_score(op_o, sc.fc, sc.cc, sc.wh, pyr[0][0], pyr[1][0], pyr[2][0], 1, 1, pb, pr, pf)
    op = ict.OptParam.from_buffer_copy(bytes(op_o))
    fr = ict.Frames(3, 320, 240, 2, 8)
    fr.upload(0, np.stack(frames))
    tr = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
    tr.set_points(np.array([0, n]), sc.points(1, n, 8, 2))
    got = tr.ncc_score(fr, 0, 1, 2, 1, 1, pb, pr, pf)
    assert (ref == -1).any() and (ref > 0.5).any()
    assert np.array_equal(got == -1, ref == -1)
    assert np.abs(got - ref).max() < 2e-5


TEACHER = [
    # dp_tol: delta_p = H^-1 J^T r inherits the J^T r error (~1e-6 of sum|sd*r|, while J^T r itself is a small difference
    # of large terms) times the conditioning of H, and the fast mode's H comes from tree sums too; measured on B200:
    # 1.4e-3 / 7.1e-3 / 3.6e-2 / 9.6e-4 of the level's first step.  The oracle's own delta_p moves as much when only
    # its Eigen packet width changes (tests/test_oracle_golden.py::test_oracle_modes_spread).  Gates = measured x 3.
    # BASELINE configs[0]/[1] geometry: 8x8 patches, 100 points, 640x480 (K2v8)
    dict(name="C1", kw=dict(seed=201, w=640, h=480, psz=8, npts=100, ntracks=4), dp_tol=5e-3),
    # BASELINE configs[2] geometry, well conditioned: 32x32 patches, 16 points per track (K2v2, one CTA of 32 warps)
    dict(name="C3-16", kw=dict(seed=202, w=1280, h=704, psz=32, npts=16, ntracks=4), dp_tol=2e-2),
    # ... and the benchmark's own ill-conditioned 4-point tracks
    dict(name="C3-4", kw=dict(seed=203, w=1280, h=704, psz=32, npts=4, ntracks=16), dp_tol=1e-1),
    # BASELINE configs[3] geometry: dense, one point per pixel (fused dense kernels), tilted plane
    dict(name="C4", kw=dict(seed=204, w=320, h=240, lv_f=2, psz=1, dense_border=8, tilt=(0.1, -0.08)), dp_tol=3e-3),
]


@pytest.mark.parametrize("tc", TEACHER, ids=[c["name"] for c in TEACHER])
def test_jtr_teacher_forced(ict, orc, tc):
    """north_star's per-iteration gate for the FAST MODE kernels (K2v2, K2v8, fused dense; tree sums, factorised
    J^T r, per-level solve matrix): the oracle's pose is forced into every iteration (ict_tracker_set_teacher), so both
    sides evaluate every J^T r and delta_p on identical inputs; J^T r must agree within 1e-5 of sum|sd*r| at EVERY
    iteration, not only the first (odometer.cpp:344-419); delta_p is gated per case (TEACHER above)."""
    from helpers import teacher_from_oracle, teacher_forced_errors
    case = make_case(**tc["kw"])
    cap = 48
    o = oracle_run(orc, case, trace_cap=cap)
    te = teacher_from_oracle(o, np.zeros((case["T"], 6)), cap)
    g = gpu_run(ict, case, trace_cap=cap, sum_order=0, teacher=te)
    jtr, dp, nrec = teacher_forced_errors(g, o)
    assert nrec >= 8 * case["T"]
    print("teacher-forced %s: %d records, worst J^T r error %.2e of sum|sd*r|, worst delta_p error %.2e of the level's first step"
          % (tc["name"], nrec, jtr, dp))
    assert jtr <= 1e-5, (tc["name"], jtr, dp)
    assert dp <= tc["dp_tol"], (tc["name"], jtr, dp)
    # forced all the way: the final pose is the oracle's last forced pose, the iteration counts are the oracle's
    assert np.array_equal(g["iters"], o["iters"])


# psz 32 has its own kernels (K2v2 for the default order, K2x for the reference order): their edge cases
CASES32 = [
    dict(seed=61, npts=1),                                   # one point: rank(H) <= 2, Eigen's truncated solve
    dict(seed=62, npts=3, ntracks=5),                        # 24 tiles: the last round of K2x is partial
    dict(seed=63, npts=7, ntracks=3),                        # 56 tiles = 8 full rounds; two groups per warp in K2v2
    dict(seed=64, npts=9, maxpttrack=6, ntracks=2),          # more points than maxpttrack
    dict(seed=65, npts=4, scale=3.0, ntracks=16),            # large motion: points leave the new frame
    dict(seed=66, npts=5, donorm=1, ntracks=4),
    dict(seed=67, npts=4, lv_f=2, lv_l=1, maxiter=3, ratio=0.1, ntracks=4),
    dict(seed=68, npts=4, maxiter=1, ntracks=3),             # a single iteration per level
]


@pytest.mark.parametrize("kw", CASES32, ids=[str(i) for i in range(len(CASES32))])
def test_psz32_kernels_edge_cases(ict, orc, kw):
    case = make_case(psz=32, w=1280, h=704, **kw)
    o = oracle_run(orc, case, trace_cap=48)
    gx = gpu_run(ict, case, trace_cap=48, sum_order=1)       # K2x: bit for bit
    assert np.array_equal(gx["pt2d"], o["pt2d"])
    assert_bit_identical(gx, o)
    g = gpu_run(ict, case, trace_cap=48)                     # K2v2: identical inputs -> J^T r to fp32 summation noise
    assert np.array_equal(g["pt2d"], o["pt2d"])
    res = check_parity(g, o, case, gates=False)
    assert res["jtr_first"] <= 1e-5, res
    assert np.array_equal(g["trace"][:, 0, 15], o["trace"][:, 0, 15])          # visible points, first iteration
    gn = gpu_run(ict, case, trace_cap=0)                     # the production instantiation (no trace records)
    assert np.array_equal(gn["p_out"], g["p_out"]) and np.array_equal(gn["iters"], g["iters"])
    assert np.array_equal(gn["npixres"], g["npixres"])


@pytest.mark.parametrize("npts", [1, 2, 4, 5, 8])
def test_k2r_equals_k2x(ict, npts):
    """The two reference-order kernels for 32x32 patches — K2r (steepest-descent images resident in shared memory, 2-D
    TMA windows; the default route) and K2x (producer/chain ring; tracker knob "no_k2r") — agree bit for bit: every
    iteration's J^T r and delta_p, iteration counts, pixel-residual counts, poses.  1..4 points run K2r with four
    producer warps, 5..8 with eight."""
    case = make_case(psz=32, w=1280, h=704, seed=160 + npts, npts=npts, ntracks=24, scale=1.5)
    c = case
    op = ict.OptParam.from_buffer_copy(bytes(c["op"]))
    fr = ict.Frames(2, c["w"], c["h"], c["lv_f"], c["psz"])
    fr.upload(0, np.stack([c["A"], c["B"]]))
    tr = ict.Tracker(op, c["sc"].fc, c["sc"].cc, c["sc"].wh)          # reference order is the library default
    tr.set_points(c["pt_off"], c["pts"].copy())
    r = tr.track_batch(fr, 0, 1, np.zeros((c["T"], 6)), trace_cap=48)
    tr.set_knob("no_k2r", 1)
    x = tr.track_batch(fr, 0, 1, np.zeros((c["T"], 6)), trace_cap=48)
    assert np.array_equal(r["trace"][..., :16], x["trace"][..., :16])
    assert np.array_equal(r["p_out"], x["p_out"]) and np.array_equal(r["iters"], x["iters"])
    assert np.array_equal(r["npixres"], x["npixres"])
    tr.close(); fr.close()


def test_psz32_kernels_points_out_of_view(ict, orc):
    """An initial pose that moves a part of the points out of the reference image (template rows stay zero, the
    coefficients stale) and others out of the new frame only at some levels."""
    case = make_case(psz=32, w=1280, h=704, seed=69, npts=6, ntracks=12)
    T = case["T"]
    p_in = np.zeros((T, 6))
    p_in[:, 0] = np.linspace(0.6, 2.4, T)                    # 150 .. 600 px to the right at level 0
    p_in[:, 4] = 0.02
    o = oracle_run(orc, case, trace_cap=48, p_in=p_in)
    assert (o["trace"][:, 0, 15] < 6).any() and (o["trace"][:, 0, 15] > 0).any()   # some, not all, points visible
    gx = gpu_run(ict, case, trace_cap=48, sum_order=1, p_in=p_in)
    assert np.array_equal(gx["pt2d"], o["pt2d"])
    assert_bit_identical(gx, o)
    g = gpu_run(ict, case, trace_cap=48, p_in=p_in)
    res = check_parity(g, o, case, gates=False)
    assert res["jtr_first"] <= 1e-5, res
    assert np.array_equal(g["trace"][:, 0, 15], o["trace"][:, 0, 15])


# psz 8 in the default order runs K2v8 (8 warps up to 128 points per track, 16 warps up to 240; with or without
# dopatchnorm)
CASES8 = [
    dict(seed=71, npts=1),                                   # one point: rank-deficient H, Eigen's truncated solve
    dict(seed=72, npts=13, ntracks=5),                       # warps with one and with two points
    dict(seed=73, npts=128, ntracks=2),                      # all sixteen point slots of every warp
    dict(seed=74, npts=130, ntracks=2),                      # K2v8 with sixteen warps, nine point slots each
    dict(seed=75, npts=90, maxpttrack=40, ntracks=2),        # more points than maxpttrack
    dict(seed=76, npts=50, scale=3.0, ntracks=6),            # large motion
    dict(seed=77, npts=60, donorm=1, dopatchnorm=1, ntracks=4),   # the MATLAB harness's settings
    dict(seed=78, npts=33, dopatchnorm=1, lv_f=2, lv_l=1, maxiter=3, ratio=0.1, ntracks=3),
    dict(seed=79, npts=200, dopatchnorm=1, ntracks=2),       # 29 rounds of seven patches, 202 KB of shared memory
    dict(seed=80, npts=230, ntracks=1),                      # beyond one CTA in the reference order: multi-CTA path
    dict(seed=81, npts=240, donorm=1, dopatchnorm=1, ntracks=1),   # K2v8's largest track (223 KB of shared memory)
]


@pytest.mark.parametrize("kw", CASES8, ids=[str(i) for i in range(len(CASES8))])
def test_psz8_kernel_edge_cases(ict, orc, kw):
    case = make_case(psz=8, **kw)
    o = oracle_run(orc, case, trace_cap=48)
    gx = gpu_run(ict, case, trace_cap=48, sum_order=1)       # K2x8 (k_track<8,2|3> beyond 224 points): bit for bit
    assert np.array_equal(gx["pt2d"], o["pt2d"])
    assert_bit_identical(gx, o)
    g = gpu_run(ict, case, trace_cap=48)
    assert np.array_equal(g["pt2d"], o["pt2d"])
    res = check_parity(g, o, case, gates=False)
    assert res["jtr_first"] <= 1e-5, res
    assert np.array_equal(g["trace"][:, 0, 15], o["trace"][:, 0, 15])          # visible points, first iteration
    if kw["npts"] >= 13:                                     # enough points for a well-conditioned problem
        assert np.abs(g["p_out"] - o["p_out"]).max() < 2e-3, res
    gn = gpu_run(ict, case, trace_cap=0)                     # the production instantiation (no trace records)
    assert np.array_equal(gn["p_out"], g["p_out"]) and np.array_equal(gn["iters"], g["iters"])
    assert np.array_equal(gn["npixres"], g["npixres"])
    gg = gpu_run(ict, case, trace_cap=48, sum_order=2)       # the general kernel in the same (tree) order class
    assert np.array_equal(gg["trace"][:, 0, 15], g["trace"][:, 0, 15])
    assert np.abs(gg["trace"][:, 0, 2:8] - g["trace"][:, 0, 2:8]).max() <= 1e-5 * np.abs(o["trace"][:, 0, 16:22]).max()


@pytest.mark.parametrize("npts", [40, 150])      # K2v8 with eight and with sixteen warps
def test_psz8_kernel_points_out_of_view(ict, orc, npts):
    case = make_case(psz=8, seed=79, npts=npts, ntracks=10)
    T = case["T"]
    p_in = np.zeros((T, 6))
    p_in[:, 0] = np.linspace(0.5, 2.2, T)
    p_in[:, 4] = 0.02
    o = oracle_run(orc, case, trace_cap=48, p_in=p_in)
    assert (o["trace"][:, 0, 15] < npts).any() and (o["trace"][:, 0, 15] > 0).any()
    assert_bit_identical(gpu_run(ict, case, trace_cap=48, sum_order=1, p_in=p_in), o)
    g = gpu_run(ict, case, trace_cap=48, p_in=p_in)
    res = check_parity(g, o, case, gates=False)
    assert res["jtr_first"] <= 1e-5, res
    assert np.array_equal(g["trace"][:, 0, 15], o["trace"][:, 0, 15])


def test_full_size_batch_properties(ict, orc):
    """BASELINE config 3 at full size (4096 four-point 32x32 tracks on one 1080p pair): size-independent properties of
    the production path — a track's result does not depend on its position in the batch, on the batch it is in, or on
    the run (bit for bit), and a sample agrees with the oracle like the small
    batches do (bit-identical in reference order)."""
    case = make_case(seed=91, w=1920, h=1080, psz=32, npts=4, ntracks=4096)
    T, P = case["T"], case["npts"]
    op = ict.OptParam.from_buffer_copy(bytes(case["op"]))
    fr = ict.Frames(2, case["w"], case["h"], case["lv_f"], case["psz"])
    fr.upload(0, np.stack([case["A"], case["B"]]))

    def run(order, sum_order=0):
        tr = ict.Tracker(op, case["sc"].fc, case["sc"].cc, case["sc"].wh)
        tr.set_sum_order(sum_order)
        pts = case["pts"].reshape(T, 3 * P)[order].reshape(-1).copy()
        tr.set_points(np.arange(len(order) + 1, dtype=np.int64) * P, pts)
        out = tr.track_batch(fr, 0, 1, np.zeros((len(order), 6)))
        tr.close()
        return out

    ident = np.arange(T)
    a = run(ident)
    b = run(ident)                                           # determinism
    assert np.array_equal(a["p_out"], b["p_out"]) and np.array_equal(a["iters"], b["iters"])
    perm = np.random.default_rng(5).permutation(T)           # position in the batch
    c = run(perm)
    assert np.array_equal(c["p_out"], a["p_out"][perm]) and np.array_equal(c["iters"], a["iters"][perm])
    assert np.array_equal(c["npixres"], a["npixres"][perm])
    h1, h2 = run(ident[:1500]), run(ident[1500:])            # the batch a track is in
    assert np.array_equal(np.concatenate([h1["p_out"], h2["p_out"]]), a["p_out"])
    # (recovering the ground-truth motion is not a property of this workload: a third of the 4-point Hessians are
    # rank-deficient by Eigen's threshold and the reference's truncated solve then leaves pose components untouched)
    # a sample of 64 tracks against the oracle: reference order bit for bit, default order on identical inputs
    sub = ident[::64]
    sc = dict(case, pts=case["pts"].reshape(T, 3 * P)[sub].reshape(-1).copy(),
              pt_off=np.arange(len(sub) + 1, dtype=np.int64) * P, T=len(sub))
    o = oracle_run(orc, sc, trace_cap=0)
    x = run(sub, sum_order=1)
    assert np.array_equal(x["p_out"], o["p_out"]) and np.array_equal(x["iters"], o["iters"])
    assert np.array_equal(x["npixres"], o["npixres"])
    xs = run(ident, sum_order=1)                             # ... and the sample is the same inside the full batch
    assert np.array_equal(xs["p_out"][sub], x["p_out"])
    assert np.median(np.abs(a["p_out"][sub] - o["p_out"]).max(axis=1)) < 1e-4   # default order: same poses in the median
    fr.close()


def test_stream_entry_points_equal_blocking_ones(ict):
    """ict_frames_upload_u8_stream / ict_tracker_set_points_stream / ict_track_batch_stream (pinned host buffers,
    copies on internal lanes, kernels on the caller's stream) give the results of the blocking entry points, chunk by
    chunk and across repeated steps that reuse the staging areas."""
    import ctypes as C
    import torch
    case = make_case(seed=95, w=1280, h=704, psz=32, npts=4, ntracks=600)
    T, P, L = case["T"], case["npts"], case["lv_f"] + 1
    op = ict.OptParam.from_buffer_copy(bytes(case["op"]))
    frames_u8 = np.stack([case["A"], case["B"]]).astype(np.uint8)
    fr = ict.Frames(2, case["w"], case["h"], case["lv_f"], case["psz"])
    fr.upload(0, frames_u8.astype(np.float32))
    tr = ict.Tracker(op, case["sc"].fc, case["sc"].cc, case["sc"].wh)
    tr.set_points(case["pt_off"], case["pts"].copy())
    ref = tr.track_batch(fr, 0, 1, np.zeros((T, 6)))
    tr.close()
    lib, v = ict.lib(), C.c_void_p
    st = torch.cuda.Stream()
    h_frames = torch.from_numpy(frames_u8).pin_memory()
    h_pts = torch.from_numpy(case["pts"].copy()).pin_memory()
    h_ref = torch.zeros(T, dtype=torch.int32).pin_memory()
    h_new = torch.ones(T, dtype=torch.int32).pin_memory()
    h_pin = torch.zeros(T, 6, dtype=torch.float64).pin_memory()
    h_pout = torch.zeros(T, 6, dtype=torch.float64).pin_memory()
    h_iters = torch.zeros(T, L, dtype=torch.int32).pin_memory()
    h_npix = torch.zeros(T, dtype=torch.int64).pin_memory()
    bounds = [0, 250, 600]
    fr2 = ict.Frames(2, case["w"], case["h"], case["lv_f"], case["psz"])
    trk = [ict.Tracker(op, case["sc"].fc, case["sc"].cc, case["sc"].wh) for _ in range(2)]
    offs = [torch.from_numpy(np.arange(bounds[c + 1] - bounds[c] + 1, dtype=np.int64) * P).pin_memory() for c in range(2)]
    for step in range(3):
        h_pout.zero_()
        for c in range(2):
            t0, t1 = bounds[c], bounds[c + 1]
            rc = lib.ict_frames_upload_u8_stream(fr2.h_, 0, 2, v(h_frames.data_ptr()), v(st.cuda_stream))
            rc |= lib.ict_tracker_set_points_stream(trk[c].h_, t1 - t0, v(offs[c].data_ptr()),
                                                    v(h_pts.data_ptr() + 8 * 3 * P * t0), v(st.cuda_stream))
            rc |= lib.ict_track_batch_stream(trk[c].h_, fr2.h_, v(h_ref.data_ptr() + 4 * t0), v(h_new.data_ptr() + 4 * t0),
                                             v(h_pin.data_ptr() + 48 * t0), v(h_pout.data_ptr() + 48 * t0),
                                             v(h_iters.data_ptr() + 4 * L * t0), v(h_npix.data_ptr() + 8 * t0),
                                             v(st.cuda_stream))
            assert rc == 0, lib.ict_last_error()
        st.synchronize()
        assert np.array_equal(h_pout.numpy(), ref["p_out"]), step
        assert np.array_equal(h_iters.numpy(), ref["iters"]) and np.array_equal(h_npix.numpy(), ref["npixres"])
    # ict_track_batch_stream after a BLOCKING ict_tracker_set_points and after ict_tracker_set_points_dev: the points'
    # copy lane was never started by those calls, the stream call has to cope (round-1 advisor finding)
    tb = ict.Tracker(op, case["sc"].fc, case["sc"].cc, case["sc"].wh)
    tb.set_points(case["pt_off"], case["pts"].copy())
    h_ref0 = torch.zeros(T, dtype=torch.int32).pin_memory()
    for variant in ("blocking", "dev"):
        if variant == "dev":
            d_off = torch.from_numpy(case["pt_off"]).cuda()
            d_pts = torch.from_numpy(case["pts"].copy()).cuda()
            tb.set_points_dev(T, d_off.data_ptr(), d_pts.data_ptr(), T * P, P)
            torch.cuda.synchronize()
        h_pout.zero_()
        rc = lib.ict_track_batch_stream(tb.h_, fr.h_, v(h_ref0.data_ptr()), v(h_new.data_ptr()), v(h_pin.data_ptr()),
                                        v(h_pout.data_ptr()), v(h_iters.data_ptr()), v(h_npix.data_ptr()), v(st.cuda_stream))
        assert rc == 0, (variant, lib.ict_last_error())
        st.synchronize()
        assert np.array_equal(h_pout.numpy(), ref["p_out"]), variant
        assert np.array_equal(h_iters.numpy(), ref["iters"]), variant
    # a frame index beyond the store is refused before anything is enqueued
    h_bad = torch.full((T,), 7, dtype=torch.int32).pin_memory()
    rc = lib.ict_track_batch_stream(tb.h_, fr.h_, v(h_ref0.data_ptr()), v(h_bad.data_ptr()), v(h_pin.data_ptr()),
                                    v(h_pout.data_ptr()), v(h_iters.data_ptr()), v(h_npix.data_ptr()), v(st.cuda_stream))
    assert rc == 2
    tb.close()
    for t_ in trk:
        t_.close()
    fr.close()
    fr2.close()


def test_robustness_modes_against_ground_truth(ict):
    """SURVEY.md §8(f4): the opt-in robustness modes (ict_tracker_set_robust; fast mode, psz 8) are judged against the
    GROUND-TRUTH motion, not against the reference whose quirks they remove.  Measured on B200
    (profiles/tools/robust_probe.py): FULL_STEP reaches the same accuracy in about half the iterations (31 -> 17 per
    track); FLOOR cuts the translation error 3x when the template centres are integer pixels >= 256, where the
    reference's ceil(x + 1e-5f) places the patch one pixel off; COMPOSE changes nothing measurable at inter-frame
    rotations of ~0.01-0.03 rad (it must not hurt)."""
    from invcompcamtrack_b200 import synth
    from invcompcamtrack_b200.api import ROBUST_FULL_STEP, ROBUST_COMPOSE, ROBUST_FLOOR, IctError

    def run(sc, A, B, pts, npts, T, flags, maxiter=10, lv_f=3, ratio=0.01, order=0):
        op = ict.make_optparam(lv_f=lv_f, lv_l=0, psz=8, maxiter=maxiter, normdp_ratio=ratio, maxpttrack=npts)
        fr = ict.Frames(2, sc.w, sc.h, lv_f, 8)
        fr.upload(0, np.stack([A, B]))
        tr = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
        tr.set_sum_order(order)
        tr.set_robust(flags)
        tr.set_points(np.arange(T + 1, dtype=np.int64) * npts, pts.copy())
        try:
            return tr.track_batch(fr, 0, 1, np.zeros((T, 6)))
        finally:
            tr.close(); fr.close()

    def terr(r, p_gt):
        return float(np.median([np.linalg.norm(p[:3] - p_gt[:3]) for p in r["p_out"]]))

    sc, A, B, p_gt = synth.make_pair(77, 640, 480)
    T, npts = 16, 100
    pts = np.concatenate([sc.points(500 + t, npts, 8, 3) for t in range(T)])
    base = run(sc, A, B, pts, npts, T, 0)
    full = run(sc, A, B, pts, npts, T, ROBUST_FULL_STEP)
    comp = run(sc, A, B, pts, npts, T, ROBUST_COMPOSE)
    assert full["iters"].sum() <= 0.65 * base["iters"].sum()           # full Gauss-Newton steps: about half the iterations
    assert terr(full, p_gt) <= 1.1 * terr(base, p_gt) and terr(base, p_gt) < 2e-3
    assert terr(comp, p_gt) <= 1.05 * terr(base, p_gt)                 # composition: no loss (and no gain at these rotations)
    # integer template centres >= 256 at level 0
    sc, A, B, p_gt = synth.make_pair(78, 640, 480)
    rng = np.random.default_rng(1)
    T, npts = 8, 64
    pts = np.concatenate([sc.backproject(rng.integers(260, 600, npts).astype(np.float64),
                                         rng.integers(260, 440, npts).astype(np.float64)) for _ in range(T)])
    ref = run(sc, A, B, pts, npts, T, 0, lv_f=0, maxiter=30, ratio=1e-3)
    flo = run(sc, A, B, pts, npts, T, ROBUST_FLOOR, lv_f=0, maxiter=30, ratio=1e-3)
    assert terr(flo, p_gt) <= 0.5 * terr(ref, p_gt)
    # the modes are not parity: the reference-order path refuses them
    with pytest.raises(IctError):
        run(sc, A, B, pts, npts, T, ROBUST_FULL_STEP, order=1)


EXTREME = [
    dict(psz=32, w=1280, h=704, npts=4, ntracks=10),     # K2r / K2v2
    dict(psz=8, npts=60, ntracks=10),                    # K2x8 / K2v8
    dict(psz=16, npts=9, ntracks=10),                    # general kernel / k_track_fast
]


@pytest.mark.parametrize("kw", EXTREME, ids=["psz32", "psz8", "psz16"])
def test_extreme_poses_stay_in_bounds(ict, orc, kw):
    """Poses that throw the patch centres far outside the padded planes, behind the camera or to infinity: the
    visibility test (odometer.cpp:369-371) must keep every placement inside the planes.  compute-sanitizer is closed on
    this pool, so the check is behavioural: reference order bit-identical to the oracle (an out-of-bounds read would
    have to return the oracle's values), both orders deterministic across runs, well-formed outputs, and an ordinary
    batch run right afterwards on the same device still bit-identical."""
    case = make_case(seed=301, **kw)
    T = case["T"]
    p_in = np.zeros((T, 6))
    p_in[0, 0] = 1e6                     # a million units sideways
    p_in[1, 1] = -3e4
    p_in[2, 2] = -50.0                   # behind the camera: negative depth
    p_in[3, 2] = -1.0                    # through the camera plane (depth ~ 0 for part of the points)
    p_in[4, 3] = np.pi                   # half a turn about x
    p_in[5, 4] = 0.5 * np.pi             # quarter turn about y: depth ~ 0
    p_in[6, 5] = 3.0                     # in-plane rotation: most points leave the frame
    p_in[7, :3] = (1e20, -1e20, 1e20)    # float overflow in the projection
    p_in[8, 2] = 1e6                     # a million units away: all points on the principal point
    p_in[9, :] = (0.3, -0.2, 0.1, 0.2, -0.3, 0.1)
    o = oracle_run(orc, case, trace_cap=48, p_in=p_in)
    g1 = gpu_run(ict, case, trace_cap=48, sum_order=1, p_in=p_in)
    assert_bit_identical(g1, o)
    g1b = gpu_run(ict, case, trace_cap=48, sum_order=1, p_in=p_in)
    assert np.array_equal(g1["p_out"], g1b["p_out"], equal_nan=True)
    g0 = gpu_run(ict, case, trace_cap=48, sum_order=0, p_in=p_in)
    g0b = gpu_run(ict, case, trace_cap=48, sum_order=0, p_in=p_in)
    assert np.array_equal(g0["p_out"], g0b["p_out"], equal_nan=True) and np.array_equal(g0["iters"], g0b["iters"])
    assert (g0["iters"] >= 0).all() and (g0["iters"] <= case["op"].maxiter).all()
    assert (g0["npixres"] >= 0).all()
    # a non-finite pose entry is undefined in the reference (it would index memory with it); here: no placement at all
    p_bad = np.zeros((T, 6))
    p_bad[0, 0] = np.nan
    p_bad[1, 4] = np.inf
    for order in (1, 0):
        gb = gpu_run(ict, case, trace_cap=0, sum_order=order, p_in=p_bad)
        assert gb["npixres"][0] == 0 and gb["npixres"][1] == 0
        assert np.isfinite(gb["p_out"][2:]).all()
    # the device is still sound: an ordinary run is bit-identical to the oracle
    o2 = oracle_run(orc, case, trace_cap=48)
    g2 = gpu_run(ict, case, trace_cap=48, sum_order=1)
    assert_bit_identical(g2, o2)


@pytest.mark.parametrize("kw", [dict(npts=24, ntracks=170), dict(npts=24, ntracks=170, dopatchnorm=1, donorm=1),
                                dict(npts=110, ntracks=150)])
def test_psz8_reference_order_both_launch_forms(ict, orc, kw):
    """K2x8 runs with seven producer warps (two CTAs per SM) for batches larger than the SM count of tracks up to 100
    points, with fifteen otherwise (small batches, tracks beyond 100 points): both bit-identical to the oracle, and a
    track's result independent of which form its batch took."""
    case = make_case(seed=311, psz=8, **kw)
    o = oracle_run(orc, case, trace_cap=48)
    g = gpu_run(ict, case, trace_cap=48, sum_order=1)
    assert_bit_identical(g, o)
    sub = dict(case)
    sub["T"] = 9
    sub["pt_off"] = case["pt_off"][:10]
    sub["pts"] = case["pts"][:3 * int(case["pt_off"][9])]      # per track: X block, Y block, Z block
    gs = gpu_run(ict, sub, trace_cap=48, sum_order=1)
    assert np.array_equal(gs["p_out"], g["p_out"][:9]) and np.array_equal(gs["iters"], g["iters"][:9])


@pytest.mark.parametrize("kw", [dict(npts=20, ntracks=170), dict(npts=50, ntracks=6), dict(npts=1, ntracks=3),
                                dict(npts=33, ntracks=5, donorm=1, lv_f=2, lv_l=1, maxiter=4, ratio=0.1),
                                dict(npts=40, maxpttrack=25, ntracks=4), dict(npts=30, scale=3.0, ntracks=8)])
def test_psz16_reference_order_kernel(ict, orc, kw):
    """16x16 patches in the reference order run K2x8 with four 64-pixel tiles per patch (both launch forms): bit-identical
    to the oracle — every iteration's J^T r and delta_p, counts, poses — incl. one point (rank-deficient H), the
    maxpttrack cap, donorm with lv_l > 0 and large motion (points leaving the frame)."""
    case = make_case(seed=321, psz=16, w=960, h=544, **kw)
    o = oracle_run(orc, case, trace_cap=48)
    g = gpu_run(ict, case, trace_cap=48, sum_order=1)
    assert np.array_equal(g["pt2d"], o["pt2d"])
    assert_bit_identical(g, o)
