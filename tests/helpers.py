"""Shared case builders for the parity tests."""
import hashlib

import numpy as np

from invcompcamtrack_b200 import synth
from oracle import oracle as O


def make_case(seed, w=640, h=480, psz=8, npts=100, lv_f=3, lv_l=0, maxiter=10, ratio=0.01, donorm=0, dopatchnorm=0,
              scale=1.0, ntracks=1, maxpttrack=None, tilt=(0.0, 0.0), dense_border=None):
    """One frame pair + ntracks independent point sets.  Returns a dict with everything both sides need.
    dense_border: one track with one point per pixel inside that border (dense alignment, psz = 1)."""
    sc, A, B, p_gt = synth.make_pair(seed, w, h, motion_scale=scale, tilt=tilt)
    if dense_border is not None:
        pts = sc.dense_points(dense_border)
        npts, ntracks = pts.size // 3, 1
        op = O.make_optparam(lv_f=lv_f, lv_l=lv_l, psz=psz, maxiter=maxiter, normdp_ratio=ratio, donorm=donorm,
                             dopatchnorm=dopatchnorm, maxpttrack=npts)
        return dict(sc=sc, A=A, B=B, p_gt=p_gt, op=op, pts=pts, pt_off=np.array([0, npts], np.int64), w=w, h=h,
                    psz=psz, lv_f=lv_f, T=1, npts=npts)
    op = O.make_optparam(lv_f=lv_f, lv_l=lv_l, psz=psz, maxiter=maxiter, normdp_ratio=ratio, donorm=donorm,
                         dopatchnorm=dopatchnorm, maxpttrack=maxpttrack or npts)
    pts = np.concatenate([sc.points(seed * 131 + t, npts, psz, lv_f) for t in range(ntracks)])
    pt_off = np.arange(ntracks + 1, dtype=np.int64) * npts
    return dict(sc=sc, A=A, B=B, p_gt=p_gt, op=op, pts=pts, pt_off=pt_off, w=w, h=h, psz=psz, lv_f=lv_f, T=ntracks,
                npts=npts)


def oracle_run(orc, case, trace_cap=64, sum_mode=0, nthreads=0, p_in=None):
    """Pyramids + batch tracking with the CPU oracle."""
    c = case
    orc.set_sum_mode(sum_mode)
    pa = orc.pyramid_build(c["A"].astype(np.float32), c["lv_f"], c["psz"])
    pb = orc.pyramid_build(c["B"].astype(np.float32), c["lv_f"], c["psz"])
    T = c["T"]
    p_in = np.zeros((T, 6)) if p_in is None else p_in
    out = orc.track_batch(c["op"], c["sc"].fc, c["sc"].cc, c["sc"].wh, [pa[0], pb[0]], [pa[1], pb[1]], [pa[2], pb[2]],
                          c["pt_off"], c["pts"].copy(), np.zeros(T, np.int32), np.ones(T, np.int32), p_in,
                          trace_cap=trace_cap, nthreads=nthreads, want_pt2d=True)
    orc.set_sum_mode(0)
    out["pyr"] = (pa, pb)
    return out


def gpu_run(ict, case, trace_cap=64, p_in=None, sum_order=0, teacher=None):
    """sum_order 0 = the opt-in fast mode (tree sums), 1 = the library default (reference order), None = leave the
    library default untouched."""
    c = case
    op = ict.OptParam.from_buffer_copy(bytes(c["op"]))
    fr = ict.Frames(2, c["w"], c["h"], c["lv_f"], c["psz"])
    fr.upload(0, np.stack([c["A"], c["B"]]))
    tr = ict.Tracker(op, c["sc"].fc, c["sc"].cc, c["sc"].wh)
    if sum_order is not None:
        tr.set_sum_order(sum_order)
    pts = c["pts"].copy()
    tr.set_points(c["pt_off"], pts)
    if teacher is not None:
        tr.set_teacher(teacher)
    T = c["T"]
    p_in = np.zeros((T, 6)) if p_in is None else p_in
    out = tr.track_batch(fr, 0, 1, p_in, trace_cap=trace_cap)
    out["pt2d"] = tr.get_2dpoints()
    out["pyr"] = (fr.download(0), fr.download(1))
    tr.close()
    fr.close()
    return out


def rot_angle_between(pa, pb):
    """Angle of R_a^T R_b for two pose coefficient vectors."""
    Ra = synth.se3_exp(pa)[:3, :3]
    Rb = synth.se3_exp(pb)[:3, :3]
    c = 0.5 * (np.trace(Ra.T @ Rb) - 1)
    # acos is ill-conditioned near 1: use the skew part
    S = Ra.T @ Rb
    s = 0.5 * np.linalg.norm([S[2, 1] - S[1, 2], S[0, 2] - S[2, 0], S[1, 0] - S[0, 1]])
    return float(np.arctan2(s, c))


def check_parity(g, o, case, jtr_tol=1e-5, rot_tol=1e-5, trans_tol=1e-5, min_same_iters=0.99, min_trans_ok=0.99,
                 jtr_traj_tol=2e-3, gates=True):
    """north_star gates between a run g and an oracle run o (which must carry a trace):

      * J^T r within 1e-5 relative on IDENTICAL inputs — the first iteration of the first level, where both sides
        start from bit-identical pose, template and frames.  "Relative" is to sum_k |sd_k * pdiff| (trace[16:22]),
        the quantity fp32 summation noise scales with (SURVEY.md §7 hard part 2; J^T r itself -> 0 at convergence).
        Later iterations are compared too but against jtr_traj_tol: from the second iteration on the two sides
        evaluate J^T r at poses that already differ in the last fp32 bits, and d(J^T r) = H * d(pose) amplifies
        that (the oracle's own summation orders differ from each other by ~3e-4 there, tests/test_oracle_golden.py).
        tests/test_gpu_parity.py::test_jtr_teacher_forced checks every iteration on identical inputs instead (the
        fast-mode kernels are fed the oracle's pose after each iteration: teacher_from_oracle below).
      * identical iteration counts on >= 99 % of (track, level);
      * converged rotation within 1e-5 rad (all tracks with identical counts);
      * translation within 1e-5 relative on >= 99 % of those tracks and within 10x that on all of them.
    Returns the measured worst cases."""
    T = case["T"]
    same = (g["iters"] == o["iters"])
    frac_same = float(same.mean())
    worst_first = 0.0
    worst_traj = 0.0
    worst_rot = 0.0
    tr_err = []
    for t in range(T):
        gt_, ot_ = g["trace"][t], o["trace"][t]
        ng, no = int((gt_[:, 0] >= 0).sum()), int((ot_[:, 0] >= 0).sum())
        for k in range(min(ng, no)):
            if gt_[k, 0] != ot_[k, 0] or gt_[k, 1] != ot_[k, 1]:
                break      # iteration structure diverged (a flipped stopping decision); counted in frac_same
            scale = np.maximum(ot_[k, 16:22].astype(np.float64), 1e-30)
            d = float((np.abs(gt_[k, 2:8].astype(np.float64) - ot_[k, 2:8]) / scale).max())
            if k == 0:
                worst_first = max(worst_first, d)
            worst_traj = max(worst_traj, d)
        if same[t].all():
            worst_rot = max(worst_rot, rot_angle_between(g["p_out"][t], o["p_out"][t]))
            tn = max(np.linalg.norm(o["p_out"][t][:3]), 1e-3)
            tr_err.append(float(np.linalg.norm(g["p_out"][t][:3] - o["p_out"][t][:3]) / tn))
    tr_err = np.array(tr_err if tr_err else [0.0])
    res = dict(frac_same=frac_same, jtr_first=worst_first, jtr_traj=worst_traj, worst_rot=worst_rot,
               worst_tr=float(tr_err.max()), frac_tr_ok=float((tr_err <= trans_tol).mean()),
               median_tr=float(np.median(tr_err)))
    if gates is False:
        return res
    assert frac_same >= min_same_iters, res
    assert worst_first <= jtr_tol, res
    assert worst_traj <= jtr_traj_tol, res
    assert worst_rot <= rot_tol, res
    assert res["frac_tr_ok"] >= min_trans_ok and res["worst_tr"] <= 10 * trans_tol, res
    return res


def assert_bit_identical(g, o):
    """Reference-order mode (ict_tracker_set_sum_order(1)) against the oracle's default mode: every iteration's
    J^T r and delta_p, the iteration counts, the pixel-residual counts and the final poses must be EQUAL."""
    assert np.array_equal(g["iters"], o["iters"])
    assert np.array_equal(g["npixres"], o["npixres"])
    gt, ot = g["trace"], o["trace"]
    assert np.array_equal(gt[..., :16], ot[..., :16]), "per-iteration trace (level, it, J^T r, delta_p, normdp, nvis)"
    assert np.array_equal(g["p_out"], o["p_out"])


def check_against_oracle_spread(g, case, orc, trace_cap=64, slack=2.0):
    """Default-order GPU run vs the oracle, judged against the reference's OWN sensitivity to the order of its fp32
    sums: the oracle is run in its default order (Eigen 3.3 SSE packets) and in two other orders the unpinned Eigen
    could equally have used (AVX packets, fp64 accumulation); the GPU's distance from the default run must not
    exceed `slack` x the largest distance between those oracle runs (plus the absolute identical-input gate
    J^T r <= 1e-5 relative on the first iteration).  Returns (gpu_metrics, oracle_spread)."""
    o0 = oracle_run(orc, case, trace_cap=trace_cap, sum_mode=0)
    spread = [check_parity(oracle_run(orc, case, trace_cap=trace_cap, sum_mode=m), o0, case, gates=False) for m in (1, 2)]
    m = check_parity(g, o0, case, gates=False)
    assert m["jtr_first"] <= 1e-5, m
    flips = max(1.0 - s["frac_same"] for s in spread)
    assert 1.0 - m["frac_same"] <= slack * flips + 0.01, (m, spread)
    assert m["median_tr"] <= slack * max(s["median_tr"] for s in spread) + 1e-6, (m, spread)
    assert m["worst_rot"] <= slack * max(s["worst_rot"] for s in spread) + 1e-6, (m, spread)
    return m, spread


def teacher_from_oracle(o, p_in, trace_cap):
    """Teacher-forcing input for ict_tracker_set_teacher from an oracle run with a trace (donorm == 0): the oracle's
    fp32 pose coefficients after every iteration — cpos_p += delta_p in fp32, pose.cpp:116-129 — and whether its loop
    went on at the same level."""
    tr = o["trace"]
    T = tr.shape[0]
    te = np.zeros((T, trace_cap, 8), np.float32)
    for t in range(T):
        p = np.asarray(p_in[t], np.float64).astype(np.float32)
        n = int((tr[t, :, 0] >= 0).sum())
        assert n < trace_cap, "trace_cap too small for teacher forcing"
        for k in range(n):
            p = (p + tr[t, k, 8:14].astype(np.float32)).astype(np.float32)
            te[t, k, :6] = p
            te[t, k, 6] = 1.0 if (k + 1 < n and tr[t, k + 1, 0] == tr[t, k, 0]) else 0.0
    return te


def teacher_forced_errors(g, o):
    """Per-iteration agreement of a teacher-forced run g with the oracle o on IDENTICAL inputs at every iteration:
    worst |J^T r difference| / sum_k|sd_k * pdiff| and worst |delta_p difference|_inf relative to the first step of the
    level, |delta_p(it = 0)|_inf — the scale the reference's own stop rule measures steps against (normdp / normdp_init,
    odometer.cpp:344-346); relative to the step itself the figure is meaningless near convergence, where delta_p is the
    image of fp32 summation noise in J^T r."""
    worst_jtr, worst_dp, nrec = 0.0, 0.0, 0
    for t in range(o["trace"].shape[0]):
        gt_, ot_ = g["trace"][t], o["trace"][t]
        n = int((ot_[:, 0] >= 0).sum())
        assert int((gt_[:, 0] >= 0).sum()) == n, "teacher forcing must reproduce the oracle's iteration structure"
        for k in range(n):
            assert gt_[k, 0] == ot_[k, 0] and gt_[k, 1] == ot_[k, 1]
            scale = np.maximum(ot_[k, 16:22].astype(np.float64), 1e-30)
            worst_jtr = max(worst_jtr, float((np.abs(gt_[k, 2:8].astype(np.float64) - ot_[k, 2:8]) / scale).max()))
            dpo = ot_[k, 8:14].astype(np.float64)
            if ot_[k, 1] == 0:
                dp0 = max(np.abs(dpo).max(), 1e-30)
            worst_dp = max(worst_dp, float(np.abs(gt_[k, 8:14] - dpo).max() / dp0))
            nrec += 1
    return worst_jtr, worst_dp, nrec


def replay_models(orc, case, pyr, p_in=None):
    """evaluate_model.TrackModel of every track of a case, on the pyramids pyr = ((I, dx, dy) of A, of B) the run
    used."""
    from evaluate_model import track_models
    c = case
    pa, pb = pyr
    T = c["T"]
    p_in = np.zeros((T, 6)) if p_in is None else p_in
    return track_models(orc, c["op"], c["sc"].fc, c["sc"].cc, c["sc"].wh, [pa[0], pb[0]], [pa[1], pb[1]],
                        [pa[2], pb[2]], c["pt_off"], c["pts"], np.zeros(T, np.int32), np.ones(T, np.int32), p_in)


def check_trajectory(run, op):
    """Exact checks of a traced run against its own records, for any kernel and sum order:
      * the records of each track are levels lv_f .. lv_l in turn, the iterations of a level run 0 .. n-1 and n is
        iters[t, level]; none was cut off (a record is left free);
      * normdp (rec[14]) is delta_p's l1 norm in the reference's association;
      * each level went on exactly while keep_iterating(it + 1, normdp, normdp of iteration 0) held;
      * npixres = novals * sum of the records' visible points."""
    from evaluate_model import normdp_l1, keep_iterating
    tr, iters, npix = run["trace"], run["iters"], run["npixres"]
    T, cap = tr.shape[:2]
    for t in range(T):
        n_rec = int((tr[t, :, 0] >= 0).sum())
        assert n_rec < cap, (t, "trace_cap too small: the trace may be truncated")
        assert (tr[t, :n_rec, 0] >= 0).all() and (tr[t, n_rec:, 0] == -1).all(), t
        recs = tr[t, :n_rec]
        k = 0
        for j, lv in enumerate(range(op.lv_f, op.lv_l - 1, -1)):
            n = int(iters[t, j])
            lr = recs[k:k + n]
            k += n
            assert n >= 1 and len(lr) == n, (t, lv, n, len(lr))
            assert (lr[:, 0] == lv).all() and (lr[:, 1] == np.arange(n)).all(), (t, lv, lr[:, :2])
            for i, r in enumerate(lr):
                assert r[14] == normdp_l1(r[8:14]), (t, lv, i, r[14], r[8:14])
                assert keep_iterating(op, i + 1, r[14], lr[0, 14]) == (i + 1 < n), (t, lv, i, r[14], lr[0, 14])
        assert k == n_rec, (t, k, n_rec)
        assert int(npix[t]) == op.novals * int(recs[:, 15].astype(np.int64).sum()), (t, npix[t])


def replay_trace_cap(op):
    """A trace_cap with room for every iteration of every level and one free record."""
    return (op.lv_f - op.lv_l + 1) * op.maxiter + 1


# ---- the seeded cases on which the oracle is compared with the reference's own sources (tests/golden/vs_ref.npz) ----
REF_CASES = [dict(seed=11), dict(seed=12, donorm=1), dict(seed=13, dopatchnorm=1), dict(seed=14, psz=4, npts=64),
             dict(seed=15, psz=16, npts=12), dict(seed=16, psz=7, npts=20, donorm=1, dopatchnorm=1),
             dict(seed=17, psz=32, npts=4, w=1920, h=1080), dict(seed=18, scale=4.0)]
REF_CAMERAS = (((640, 480), (600.5, 610.25), (321.5, 239.25), 8), ((1920, 1080), (1920, 1920), (960, 540), 32))
PYR_SAMPLE = 2048          # pyramid values stored per plane beside the digest of the whole plane


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def pyramid_sample_index(n, seed):
    return np.sort(np.random.default_rng(seed).choice(n, size=min(PYR_SAMPLE, n), replace=False))


def ref_outputs(lib, orc):
    """Everything the comparison with the reference records, computed by lib (OracleLib or RefLib), as one dict of
    arrays: per case k the digest of the seeded inputs, lib's pyramid of the first frame (digest + seeded sample), and
    Set3Dpoints -> SetPose -> TrackPose on the oracle's pyramids (pose, every iteration's J^T r and delta_p, reference
    reprojection, possibly centred points); camera levels; the poses of one 12-track batch."""
    out = {}
    for k, kw in enumerate(REF_CASES):
        c = make_case(**kw)
        lv_f, psz = c["lv_f"], c["psz"]
        tot, off, sw, sh = O.pyramid_layout(c["w"], c["h"], lv_f, psz)
        pa = lib.pyramid_build(c["A"].astype(np.float32), lv_f, psz)
        pa_o = orc.pyramid_build(c["A"].astype(np.float32), lv_f, psz)
        pb_o = orc.pyramid_build(c["B"].astype(np.float32), lv_f, psz)
        od = O.Odometer(lib, c["op"], c["sc"].fc, c["sc"].cc, c["sc"].wh)
        pts = c["pts"].copy()
        od.set3dpoints(pts)
        od.setpose(np.zeros(6), pa_o, pb_o, lv_f, off)
        q = od.get2dpoints()
        if isinstance(lib, O.RefLib):
            p, sv = lib.track(od, 96)
            jtr, dp = sv[:, 36:42], sv[:, 42:48]
        else:
            p, it, tr, npx = lib.track(od, 96)
            jtr, dp = tr[:, 2:8], tr[:, 8:14]
        od.close()
        idx = pyramid_sample_index(pa[0].size, k)
        out.update({"t%d_inputs" % k: digest(c["A"], c["B"], c["pts"]), "t%d_pyr" % k: digest(*pa),
                    "t%d_pyr_sample" % k: np.stack([a[idx] for a in pa]), "t%d_p" % k: p, "t%d_jtr" % k: jtr,
                    "t%d_dp" % k: dp, "t%d_q" % k: q, "t%d_pts" % k: pts})
    for k, (wh, fc, cc, pad) in enumerate(REF_CAMERAS):
        out["camera%d" % k] = lib.camera_levels(4, fc, cc, wh, pad)
    c = make_case(seed=19, ntracks=12, npts=24)
    pa = orc.pyramid_build(c["A"].astype(np.float32), c["lv_f"], c["psz"])
    pb = orc.pyramid_build(c["B"].astype(np.float32), c["lv_f"], c["psz"])
    batch = lib.track_batch(c["op"], c["sc"].fc, c["sc"].cc, c["sc"].wh, [pa[0], pb[0]], [pa[1], pb[1]],
                            [pa[2], pb[2]], c["pt_off"], c["pts"].copy(), np.zeros(12, np.int32), np.ones(12, np.int32),
                            np.zeros((12, 6)), nthreads=2)
    out["batch_p_out"] = batch if isinstance(lib, O.RefLib) else batch["p_out"]
    return out
