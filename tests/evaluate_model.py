"""CPU model of ict_track_evaluate (test infrastructure): one Gauss-Newton measurement per track at a chosen pose,
built from the CPU oracle's pinned pieces — setpose_se3's arithmetic with the oracle's se3_exp / se3_log, its
getpatch / getpatch_grad (placement, weights, patch means), its Eigen packet sums (OracleLib.esum in the current sum
mode) and its fullPivLu solve — with every fp32 / fp64 operation in the reference's order (numpy rounds each
operation), so that its outputs are bit-identical to TrackPose's where the two measure the same thing
(tests/test_oracle_evaluate.py pins that).

    evaluate_track(orc, op, cam, pyr_ref, pyr_new, offs, sw, pts, p_ref, p_cur, level)   one track
    evaluate_batch(orc, op, fc, cc, wh, planes_I, planes_dx, planes_dy, pt_off, pts, ref_frame, new_frame, p_ref,
                   p_cur=None, level=None)                                              a batch, outputs stacked
    TrackModel(...).measure(p, level)      the same at fp32 internal pose coefficients, template cached per level
    replay_batch(...)                      a traced tracking run re-measured along its own trajectory

Outputs as include/ictrack.h defines them, plus the fp64 normalisers of the tolerance gates: habs[21] = sum|sd_a*sd_b|
(ComputeHessian's order of the pairs), jabs[6] = sum|sd_k*pdiff|, ssr_d = sum pdiff^2.
"""
import numpy as np

from oracle import oracle as O

f32, f64 = np.float32, np.float64
PAIRS = [(a, b) for a in range(6) for b in range(a, 6)]      # ComputeHessian, odometer.cpp:430-455
BORDER_PX = 1e-3     # TrackModel.measure's nborder: points whose new-frame pixel lies this close to the image bounds


def set3dpoints(op, pts):
    """OdometerClass::Set3Dpoints (odometer.cpp:171-239): the float points and (meanshift, varval); the fp64 sums are
    sequential, as there."""
    n_in = pts.size // 3
    n = min(n_in, op.maxpttrack)
    p = [np.asarray(pts[k * n_in:k * n_in + n], f64) for k in range(3)]
    if not op.donorm:
        return [x.astype(f32) for x in p], np.zeros(3), 0.0
    seq = lambda x: float(np.add.accumulate(np.concatenate([[0.0], x]))[-1])   # noqa: E731  ((0 + x0) + x1) + ...
    with np.errstate(invalid="ignore", divide="ignore"):
        ms = np.array([seq(x) for x in p]) / f64(n)
        c = [x - m for x, m in zip(p, ms)]
        var = seq(c[0] * c[0] + c[1] * c[1] + c[2] * c[2]) / f64(n)
        return [(x / var).astype(f32) for x in c], ms, var


def internal_pose(orc, p_in, donorm, ms, var):
    """PoseClass::setpose_se3 (pose.cpp:25-76): the fp32 coefficients cpos_p it keeps — p_in rounded to fp32, or with
    donorm the coefficients of the pose in the normalised point frame (se3_log in fp64, narrowed)."""
    p = np.asarray(p_in, f64).copy()
    if donorm:
        with np.errstate(invalid="ignore", divide="ignore"):
            G = orc.se3_exp(p, f64)
            t = np.array([-G[0] * G[3] - G[4] * G[7] - G[8] * G[11], -G[1] * G[3] - G[5] * G[7] - G[9] * G[11],
                          -G[2] * G[3] - G[6] * G[7] - G[10] * G[11]])
            t = (t - ms) / var
            G[3] = -G[0] * t[0] - G[1] * t[1] - G[2] * t[2]
            G[7] = -G[4] * t[0] - G[5] * t[1] - G[6] * t[2]
            G[11] = -G[8] * t[0] - G[9] * t[1] - G[10] * t[2]
            p = orc.se3_log(G, f64)
    return p.astype(f32)


def setpose_se3(orc, p_in, donorm, ms, var):
    """PoseClass::setpose_se3 (pose.cpp:25-76): the fp32 group element."""
    return orc.se3_exp(internal_pose(orc, p_in, donorm, ms, var), f32)


def getpose_se3(orc, p, donorm, ms, var):
    """PoseClass::getPose_se3 (pose.cpp:79-113) of the fp32 coefficients p (G = se3_exp_f(p), as TrackPose keeps it):
    the pose in the caller's point frame, as float64."""
    p = np.asarray(p, f32)
    if not donorm:
        return p.astype(f64)
    G = orc.se3_exp(p, f32)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        t = np.array([f64(-G[0] * G[3] - G[4] * G[7] - G[8] * G[11]), f64(-G[1] * G[3] - G[5] * G[7] - G[9] * G[11]),
                      f64(-G[2] * G[3] - G[6] * G[7] - G[10] * G[11])])    # fp32 expressions, widened
        t = t * var + ms
        g = G.astype(f64)
        G[3] = f32(-g[0] * t[0] - g[1] * t[1] - g[2] * t[2])
        G[7] = f32(-g[4] * t[0] - g[5] * t[1] - g[6] * t[2])
        G[11] = f32(-g[8] * t[0] - g[9] * t[1] - g[10] * t[2])
    return orc.se3_log(G, f32).astype(f64)


def normdp_l1(dp):
    """delta_p.lpNorm<1>() (odometer.cpp:412) in fp32, Eigen 3.3's association."""
    a = np.abs(np.asarray(dp, f32))
    return ((a[0] + a[2]) + (a[1] + a[3])) + (a[4] + a[5])


def keep_iterating(op, done, normdp, normdp_init):
    """The stop rule (odometer.cpp:341-346) after `done` iterations of a level, fp32 division."""
    with np.errstate(invalid="ignore", divide="ignore"):
        return bool((done < op.maxiter) & ((f32(normdp) / f32(normdp_init)) > f32(op.normdp_ratio)))


def project(G, X, Y, Z, cam, l):
    """project_pt (pose.cpp:307-397) at level l, fp32; returns the camera-frame point and the pixel."""
    with np.errstate(invalid="ignore", divide="ignore"):
        tx = G[0] * X + G[1] * Y + G[2] * Z + G[3]
        ty = G[4] * X + G[5] * Y + G[6] * Z + G[7]
        tz = G[8] * X + G[9] * Y + G[10] * Z + G[11]
        return (tx, ty, tz), (tx / tz) * f32(cam[l, 0]) + f32(cam[l, 2]), (ty / tz) * f32(cam[l, 1]) + f32(cam[l, 3])


def inside(x, y, cam, l):
    """odometer.cpp:273-275 / 369-371, written so that NaN is outside."""
    return (x >= 0) & (y >= 0) & (x <= f32(cam[l, 4])) & (y <= f32(cam[l, 5]))


def sd_images(dx, dy, xc, yc, zc, fx, fy):
    """odometer.cpp:306-326 for one point: the six steepest-descent values of its pixels."""
    zsq = zc * zc
    c1x, c2y = fx / zc, fy / zc
    c3x, c3y = (-xc) / zsq * fx, (-yc) / zsq * fy
    c4x = (-xc) * yc / zsq * fx
    c4y = f32((-(1.0 + f64(yc * yc / zsq))) * f64(fy))
    c5x = f32((1.0 + f64(xc * xc / zsq)) * f64(fx))
    c5y = xc * yc / zsq * fy
    c6x, c6y = (-yc) / zc * fx, xc / zc * fy
    return [dx * c1x, dy * c2y, dx * c3x + dy * c3y, dx * c4x + dy * c4y, dx * c5x + dy * c5y, dx * c6x + dy * c6y]


class TrackModel:
    """One track of TrackPose split the way the kernels split it: what depends on the SetPose pose only — the points,
    the internal pose p0, and per level the template (placement, getpatch_grad, steepest-descent values) and its
    Hessian — is built once and cached; measure() redoes only the new image's side at a pose."""

    def __init__(self, orc, op, cam, pyr_ref, pyr_new, offs, sw, pts, p_ref):
        self.orc, self.op, self.cam, self.offs, self.sw = orc, op, cam, offs, sw
        self.pyr_ref, self.pyr_new = pyr_ref, pyr_new
        self.n_in = pts.size // 3
        (self.X, self.Y, self.Z), self.ms, self.var = set3dpoints(op, pts)
        self.p0 = internal_pose(orc, p_ref, op.donorm, self.ms, self.var)
        self.Gr = orc.se3_exp(self.p0, f32)
        self.ref3 = project(self.Gr, self.X, self.Y, self.Z, cam, op.lv_f)[0]
        self._levels = {}

    def plane(self, a, l):
        return a[self.offs[l]:]

    def internal(self, p_in):
        """SetPose's internal coefficients of another pose in this track's point frame."""
        return internal_pose(self.orc, p_in, self.op.donorm, self.ms, self.var)

    def getpose(self, p):
        return getpose_se3(self.orc, p, self.op.donorm, self.ms, self.var)

    def level(self, level):
        """(template, sd[6], H, habs) at `level`: TrackPose keeps a point's slots of the last level, walking down from
        lv_f, at which it was inside the reference image."""
        if level in self._levels:
            return self._levels[level]
        op, orc, cam = self.op, self.orc, self.cam
        M, nv, P = op.maxpttrack, op.novals, self.X.size
        if level == op.lv_f:
            tmpl, sd = np.zeros((M, nv), f32), np.zeros((6, M, nv), f32)
        else:
            tmpl, sd, _, _ = self.level(level + 1)
            tmpl, sd = tmpl.copy(), sd.copy()
        _, x, y = project(self.Gr, self.X, self.Y, self.Z, cam, level)
        vis = inside(x, y, cam, level)
        xc, yc, zc = self.ref3
        for i in range(P):
            if vis[i]:
                I, dx, dy = orc.getpatch_grad(self.plane(self.pyr_ref[0], level), self.plane(self.pyr_ref[1], level),
                                              self.plane(self.pyr_ref[2], level), [x[i], y[i]], op, self.sw[level])
                tmpl[i] = I
                s = sd_images(dx, dy, xc[i], yc[i], zc[i], f32(cam[level, 0]), f32(cam[level, 1]))
                for k in range(6):
                    sd[k, i] = s[k]
        sdf = sd.reshape(6, -1)
        H = np.zeros((6, 6), f32)
        habs = np.zeros(21)
        for q, (a, b) in enumerate(PAIRS):
            prod = sdf[a] * sdf[b]
            H[a, b] = H[b, a] = orc.esum(prod)
            habs[q] = np.abs(prod.astype(f64)).sum()
        self._levels[level] = (tmpl, sd, H, habs)
        return self._levels[level]

    def measure(self, p, level, per_point=True):
        """One iteration's measurement at the fp32 internal coefficients p (G = se3_exp_f(p)).  nborder counts the
        points whose new-frame pixel lies within BORDER_PX of the bounds (their visibility is a rounding away from
        flipping); pt_ssr / ssr only with per_point."""
        op, orc, cam = self.op, self.orc, self.cam
        M, nv, P = op.maxpttrack, op.novals, self.X.size
        tmpl, sd, H, habs = self.level(level)
        G = orc.se3_exp(np.asarray(p, f32), f32)
        _, nx, ny = project(G, self.X, self.Y, self.Z, cam, level)
        vis_new = inside(nx, ny, cam, level)
        with np.errstate(invalid="ignore"):
            edge = np.minimum.reduce([np.abs(nx), np.abs(ny), np.abs(nx - f32(cam[level, 4])),
                                      np.abs(ny - f32(cam[level, 5]))])
        pd = np.zeros((M, nv), f32)
        pt_ssr = np.full(self.n_in, -1.0, f32)
        for i in np.flatnonzero(vis_new):
            new = orc.getpatch(self.plane(self.pyr_new[0], level), [nx[i], ny[i]], op, self.sw[level])
            pd[i] = tmpl[i] - new
            if per_point:
                pt_ssr[i] = orc.esum(pd[i] * pd[i])
        sdf, pdf = sd.reshape(6, -1), pd.reshape(-1)
        jp = sdf * pdf
        jtr = np.array([orc.esum(jp[k]) for k in range(6)], f32)
        out = dict(H=H, jtr=jtr, dp=orc.solve6(H, jtr), nvis=int(vis_new.sum()), nborder=int((edge < BORDER_PX).sum()),
                   habs=habs, jabs=np.abs(jp.astype(f64)).sum(1))
        if per_point:
            out.update(ssr=f32(orc.esum(pdf * pdf)), pt_ssr=pt_ssr, ssr_d=float((pdf.astype(f64) ** 2).sum()))
        return out


def evaluate_track(orc, op, cam, pyr_ref, pyr_new, offs, sw, pts, p_ref, p_cur, level):
    m = TrackModel(orc, op, cam, pyr_ref, pyr_new, offs, sw, pts, p_ref)
    return m.measure(m.p0 if p_cur is None else m.internal(p_cur), level)


def batch_geometry(orc, op, fc, cc, wh):
    cam = orc.camera_levels(op.lv_f + 1, fc, cc, wh, op.psz)
    _, offs, sw, _ = O.pyramid_layout(int(wh[0]), int(wh[1]), op.lv_f, op.psz)
    return cam, offs, sw


def track_models(orc, op, fc, cc, wh, planes_I, planes_dx, planes_dy, pt_off, pts, ref_frame, new_frame, p_ref):
    """One TrackModel per track of a batch over flat per-frame plane sets (one per frame, laid out as
    ict_pyramid_layout)."""
    cam, offs, sw = batch_geometry(orc, op, fc, cc, wh)
    out = []
    for t in range(len(pt_off) - 1):
        a, b = int(pt_off[t]), int(pt_off[t + 1])
        rf, nf = int(ref_frame[t]), int(new_frame[t])
        out.append(TrackModel(orc, op, cam, (planes_I[rf], planes_dx[rf], planes_dy[rf]), (planes_I[nf],), offs, sw,
                              np.asarray(pts[3 * a:3 * b], f64), p_ref[t]))
    return out


def evaluate_batch(orc, op, fc, cc, wh, planes_I, planes_dx, planes_dy, pt_off, pts, ref_frame, new_frame, p_ref,
                   p_cur=None, level=None):
    """A batch over flat per-frame plane sets; pt_ssr laid out like the points.  level defaults to lv_l."""
    level = op.lv_l if level is None else level
    keys = ("H", "jtr", "dp", "ssr", "nvis", "habs", "jabs", "ssr_d")
    out = {k: [] for k in keys}
    pt_ssr = []
    models = track_models(orc, op, fc, cc, wh, planes_I, planes_dx, planes_dy, pt_off, pts, ref_frame, new_frame, p_ref)
    for t, m in enumerate(models):
        r = m.measure(m.p0 if p_cur is None else m.internal(p_cur[t]), level)
        for k in keys:
            out[k].append(r[k])
        pt_ssr.append(r["pt_ssr"])
    res = {k: np.array(v) for k, v in out.items()}
    res["ssr"] = res["ssr"].astype(f32)
    res["nvis"] = res["nvis"].astype(np.int32)
    res["pt_ssr"] = np.concatenate(pt_ssr) if pt_ssr else np.zeros(0, f32)
    return res


def replay_track(m, trace):
    """Re-measure one track's traced run along its own trajectory.  Every tracking kernel, like TrackPose
    (pose.cpp:116-129), keeps fp32 coefficients p, starts at SetPose's p0 and after each iteration adds the delta_p it
    records: p_{k+1} = fl32(p_k + delta_p_k).  So the pose of every measurement is rebuilt exactly from the trace, and
    the model measures there.  Returns the model's records in the oracle's layout — [0..15] as include/ictrack.h,
    [16..21] jabs — the rebuilt final pose through getPose_se3, and nborder per record."""
    recs = trace[trace[:, 0] >= 0]
    out = np.zeros((trace.shape[0], O.TRACE_FLOATS), f32)
    out[len(recs):, 0] = -1
    nborder = np.zeros(len(recs), np.int64)
    p = m.p0.copy()
    for k, r in enumerate(recs):
        e = m.measure(p, int(r[0]), per_point=False)
        o = out[k]
        o[0], o[1] = r[0], r[1]
        o[2:8], o[8:14] = e["jtr"], e["dp"]
        o[14] = normdp_l1(e["dp"])
        o[15] = e["nvis"]
        o[16:22] = e["jabs"]
        nborder[k] = e["nborder"]
        p = (p + r[8:14].astype(f32)).astype(f32)
    return out, m.getpose(p), nborder


def replay_batch(models, trace):
    """replay_track over a batch: trace [T, cap, 24] -> dict(trace, p_out, nborder (one array per track))."""
    res = [replay_track(m, trace[t]) for t, m in enumerate(models)]
    return dict(trace=np.stack([r[0] for r in res]), p_out=np.array([r[1] for r in res]).reshape(-1, 6),
                nborder=[r[2] for r in res])
