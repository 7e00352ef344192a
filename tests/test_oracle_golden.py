"""CPU: pins the oracle (oracle/ictrack_oracle.c) against the committed golden fixtures:
pyramids computed with Python cv2, everything else produced by the reference's own sources (oracle/_ref), see
tests/golden/make_golden.py.  Bit-exact throughout."""
import glob
import os

import numpy as np
import pytest

from oracle import oracle as O

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("name", ["rand", "sqrt", "tex"])
def test_pyramid_matches_cv2(orc, name):
    z = np.load(os.path.join(GOLD, "pyramid_%s.npz" % name))
    I, dx, dy = orc.pyramid_build(z["img"].astype(np.float32), int(z["lv_f"]), int(z["pad"]))
    assert np.array_equal(I, z["I"])
    assert np.array_equal(dx, z["dx"])
    assert np.array_equal(dy, z["dy"])


def test_se3_exp_log_match_reference(orc):
    z = np.load(os.path.join(GOLD, "se3.npz"))
    for k, p in enumerate(z["P"]):
        assert np.array_equal(orc.se3_exp(p, np.float32), z["Gf"][k])
        assert np.array_equal(orc.se3_exp(p, np.float64), z["Gd"][k])
        assert np.array_equal(orc.se3_log(z["Gf"][k], np.float32), z["lf"][k], equal_nan=True)
        assert np.array_equal(orc.se3_log(z["Gd"][k], np.float64), z["ld"][k], equal_nan=True)


def test_getpatch_matches_reference(orc):
    z = np.load(os.path.join(GOLD, "getpatch.npz"))
    img, mids = z["img"], z["mids"]
    for psz in (8, 5, 1):
        I, dx, dy = orc.pyramid_build(img, 0, psz)
        width = img.shape[1] + 2 * psz
        for pn in (0, 1):
            op = O.make_optparam(lv_f=0, psz=psz, dopatchnorm=pn, maxpttrack=4)
            for k, m in enumerate(mids):
                assert np.array_equal(orc.getpatch(I, m, op, width), z["p%d_n%d" % (psz, pn)][k]), (psz, pn, k)
                g = orc.getpatch_grad(I, dx, dy, m, op, width)
                assert np.array_equal(np.stack(g), z["g%d_n%d" % (psz, pn)][k]), (psz, pn, k)


def test_ceil_quirk_of_patch_placement(orc):
    """SURVEY §9.2: ceil(x+1e-5f) in fp32 equals floor(x)+1 for integer x < 256 but floor(x) for integer x >= 256."""
    img = np.arange(64 * 640, dtype=np.float32).reshape(64, 640) % 251
    I, _, _ = orc.pyramid_build(img, 0, 8)
    op = O.make_optparam(lv_f=0, psz=8, maxpttrack=4)
    width = 640 + 16
    lo = orc.getpatch(I, [100.0, 20.0], op, width)       # samples columns 100-3 .. : shifted by one
    hi = orc.getpatch(I, [300.0, 20.0], op, width)
    P = I.reshape(64 + 16, width)
    assert lo[0] == P[8 + 20 - 4 + 1 - 1, 8 + 100 - 4 + 1 - 1]
    assert hi[0] == P[8 + 20 - 4 + 1 - 1, 8 + 300 - 4 - 1]


TRACKS = sorted(os.path.basename(p)[6:-4] for p in glob.glob(os.path.join(GOLD, "track_*.npz")))


@pytest.mark.parametrize("name", TRACKS)
def test_track_matches_reference(orc, name):
    """Set3Dpoints -> SetPose -> TrackPose: pose, reference reprojection, centred points and EVERY iteration's
    Hessian, J^T r and delta_p identical to the reference's own sources."""
    z = np.load(os.path.join(GOLD, "track_%s.npz" % name))
    op = O.OptParam.from_buffer_copy(z["op"].tobytes())
    A, B = z["A"], z["B"]
    lv_f, psz = op.lv_f, op.psz
    tot, off, sw, sh = O.pyramid_layout(A.shape[1], A.shape[0], lv_f, psz)
    pa = orc.pyramid_build(A.astype(np.float32), lv_f, psz)
    pb = orc.pyramid_build(B.astype(np.float32), lv_f, psz)
    od = O.Odometer(orc, op, z["fc"], z["cc"], z["wh"])
    pts = z["pts"].copy()
    od.set3dpoints(pts)
    od.setpose(z["p_in"], pa, pb, lv_f, off)
    assert np.array_equal(od.get2dpoints(), z["pt2d"], equal_nan=True)
    assert np.array_equal(pts, z["pts_after"])
    p_out, iters, trace, npix = orc.track(od, 128)
    od.close()
    solves = z["solves"]
    assert len(trace) == len(solves) == int(iters.sum())
    assert np.array_equal(trace[:, 2:8], solves[:, 36:42])
    assert np.array_equal(trace[:, 8:14], solves[:, 42:48])
    assert np.array_equal(p_out, z["p_out"])


def test_solve6_restatement_is_a_solver(orc):
    """The restated fullPivLu().solve() must at least solve SPD systems to fp32 accuracy (independent check)."""
    rng = np.random.default_rng(0)
    for _ in range(20):
        M = rng.standard_normal((6, 12))
        H = (M @ M.T).astype(np.float32)
        b = rng.standard_normal(6).astype(np.float32)
        x = orc.solve6(H, b)
        assert np.allclose(H.astype(np.float64) @ x, b, atol=5e-4 * np.abs(b).max() * np.linalg.cond(H) ** 0.5)
    # rank-deficient: Eigen's rank() zeroes the null-space part instead of dividing by ~0
    H = np.zeros((6, 6), np.float32); H[0, 0] = 4; H[1, 1] = 2
    x = orc.solve6(H, np.array([4, 2, 1, 1, 1, 1], np.float32))
    assert np.array_equal(x, np.array([1, 1, 0, 0, 0, 0], np.float32))


def test_sum_orders_agree_to_fp32_noise(orc):
    """Packet-order (Eigen 3.3 SSE / AVX), sequential and fp64-accumulate sums of the same data differ only by
    fp32 rounding; the fp64 mode is the arbiter used in the GPU tests."""
    rng = np.random.default_rng(1)
    a = (rng.standard_normal(6400) * 1e4).astype(np.float32)
    vals = []
    for m in range(4):
        orc.set_sum_mode(m)
        vals.append(orc.esum(a))
    orc.set_sum_mode(0)
    ref = float(a.astype(np.float64).sum())
    scale = float(np.abs(a).astype(np.float64).sum())
    assert abs(vals[2] - ref) <= 1e-7 * scale
    for v in vals:
        assert abs(v - ref) <= 2e-5 * scale
    assert orc.esum(np.zeros(0, np.float32)) == 0.0
    assert orc.esum(np.array([1, 2, 3], np.float32)) == 6.0


def test_oracle_recovers_ground_truth(orc):
    """The restated tracker is a tracker: it recovers the known motion of a synthetic pair."""
    from helpers import make_case, oracle_run
    case = make_case(seed=0)
    o = oracle_run(orc, case, trace_cap=0)
    assert np.abs(o["p_out"][0] - case["p_gt"]).max() < 3e-3
    assert (o["iters"] >= 2).all()      # min two iterations per level (SURVEY §9.7)


def test_oracle_modes_spread(orc):
    """How far the REFERENCE'S OWN result moves when only the order of its fp32 sums changes (Eigen SSE packets vs
    AVX packets vs fp64 accumulation): identical inputs -> J^T r within ~3e-6 of sum|sd*r|, but a few percent of the
    (track, level) stopping decisions flip and the pose moves by ~1e-5 relative.  This is the noise floor the GPU's
    tree order is judged against in tests/test_gpu_parity.py."""
    from helpers import make_case, oracle_run, check_parity
    case = make_case(seed=0, ntracks=16)
    o0 = oracle_run(orc, case, sum_mode=0)
    for mode in (1, 2):
        om = oracle_run(orc, case, sum_mode=mode)
        res = check_parity(om, o0, case, min_same_iters=0.85, min_trans_ok=0.5, jtr_traj_tol=1.0)
        assert res["jtr_first"] < 1e-5


def test_degenerate_donorm_tracks(orc):
    """donorm on a track of one point (or of equal points) divides by a variance of 0 and on an empty track by 0
    points: the points become NaN.  A NaN placement is not visible (the test reads !(x >= 0 & ... & y <= sho), as the
    kernels do), so such a track runs one iteration per level on no pixel and returns a NaN translation and a zero
    rotation; the other tracks of the batch are not affected."""
    from invcompcamtrack_b200 import synth
    sc, A, B, _ = synth.make_pair(21, 320, 240)
    pa = orc.pyramid_build(A.astype(np.float32), 2, 8)
    pb = orc.pyramid_build(B.astype(np.float32), 2, 8)
    sizes = [5, 1, 0, 37]
    pts = [sc.points(90 + t, n, 8, 2) for t, n in enumerate(sizes)]
    pt_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    op = O.make_optparam(lv_f=2, psz=8, donorm=1, maxpttrack=40)

    def run(idx):
        n = [sizes[t] for t in idx]
        return orc.track_batch(op, sc.fc, sc.cc, sc.wh, [pa[0], pb[0]], [pa[1], pb[1]], [pa[2], pb[2]],
                               np.concatenate([[0], np.cumsum(n)]).astype(np.int64),
                               np.concatenate([pts[t] for t in idx]), np.zeros(len(idx), np.int32),
                               np.ones(len(idx), np.int32), np.zeros((len(idx), 6)), trace_cap=16, want_pt2d=True)
    o = run(range(4))
    for t in (1, 2):
        assert np.isnan(o["p_out"][t, :3]).all() and np.array_equal(o["p_out"][t, 3:], np.zeros(3))
        assert np.array_equal(o["iters"][t], [1, 1, 1]) and o["npixres"][t] == 0
        assert (o["trace"][t, :3, 15] == 0).all()
    assert np.isnan(o["pt2d"][2 * pt_off[1]:2 * pt_off[2]]).all()
    for t in (0, 3):
        assert np.isfinite(o["p_out"][t]).all() and (o["iters"][t] >= 2).all()
        alone = run([t])
        assert np.array_equal(alone["p_out"][0], o["p_out"][t])
        assert np.array_equal(alone["trace"][0], o["trace"][t])
        assert np.array_equal(alone["pt2d"], o["pt2d"][2 * pt_off[t]:2 * pt_off[t + 1]])
