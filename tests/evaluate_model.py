"""CPU model of ict_track_evaluate (test infrastructure): one Gauss-Newton measurement per track at a chosen pose,
built from the CPU oracle's pinned pieces — setpose_se3's arithmetic with the oracle's se3_exp / se3_log, its
getpatch / getpatch_grad (placement, weights, patch means), its Eigen packet sums (OracleLib.esum in the current sum
mode) and its fullPivLu solve — with every fp32 / fp64 operation in the reference's order (numpy rounds each
operation), so that its outputs are bit-identical to TrackPose's where the two measure the same thing
(tests/test_oracle_evaluate.py pins that).

    evaluate_track(orc, op, cam, pyr_ref, pyr_new, offs, sw, pts, p_ref, p_cur, level)   one track
    evaluate_batch(orc, op, fc, cc, wh, planes_I, planes_dx, planes_dy, pt_off, pts, ref_frame, new_frame, p_ref,
                   p_cur=None, level=None)                                              a batch, outputs stacked

Outputs as include/ictrack.h defines them, plus the fp64 normalisers of the tolerance gates: habs[21] = sum|sd_a*sd_b|
(ComputeHessian's order of the pairs), jabs[6] = sum|sd_k*pdiff|, ssr_d = sum pdiff^2.
"""
import numpy as np

from oracle import oracle as O

f32, f64 = np.float32, np.float64
PAIRS = [(a, b) for a in range(6) for b in range(a, 6)]      # ComputeHessian, odometer.cpp:430-455


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


def setpose_se3(orc, p_in, donorm, ms, var):
    """PoseClass::setpose_se3 (pose.cpp:25-76): the fp32 group element."""
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
    return orc.se3_exp(p.astype(f32), f32)


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


def evaluate_track(orc, op, cam, pyr_ref, pyr_new, offs, sw, pts, p_ref, p_cur, level):
    n_in = pts.size // 3
    (X, Y, Z), ms, var = set3dpoints(op, pts)
    P, M, nv = X.size, op.maxpttrack, op.novals
    Gr = setpose_se3(orc, p_ref, op.donorm, ms, var)
    Gc = setpose_se3(orc, p_ref if p_cur is None else p_cur, op.donorm, ms, var)
    plane = lambda a, l: a[offs[l]:]          # noqa: E731
    tmpl = np.zeros((M, nv), f32)
    sd = np.zeros((6, M, nv), f32)
    pd = np.zeros((M, nv), f32)
    pt_ssr = np.full(n_in, -1.0, f32)
    (xc, yc, zc), _, _ = project(Gr, X, Y, Z, cam, op.lv_f)
    lvl = np.full(P, -1)
    for l in range(op.lv_f, level - 1, -1):   # TrackPose keeps a point's slots of the last level it was inside at
        _, x, y = project(Gr, X, Y, Z, cam, l)
        lvl[inside(x, y, cam, l)] = l
    nvis = 0
    _, nx, ny = project(Gc, X, Y, Z, cam, level)
    vis_new = inside(nx, ny, cam, level)
    for i in range(P):
        if lvl[i] >= 0:
            l = lvl[i]
            _, x, y = project(Gr, X[i:i + 1], Y[i:i + 1], Z[i:i + 1], cam, l)
            I, dx, dy = orc.getpatch_grad(plane(pyr_ref[0], l), plane(pyr_ref[1], l), plane(pyr_ref[2], l),
                                          [x[0], y[0]], op, sw[l])
            tmpl[i] = I
            s = sd_images(dx, dy, xc[i], yc[i], zc[i], f32(cam[l, 0]), f32(cam[l, 1]))
            for k in range(6):
                sd[k, i] = s[k]
        if vis_new[i]:
            nvis += 1
            new = orc.getpatch(plane(pyr_new[0], level), [nx[i], ny[i]], op, sw[level])
            pd[i] = tmpl[i] - new
            pt_ssr[i] = orc.esum(pd[i] * pd[i])
    sdf, pdf = sd.reshape(6, -1), pd.reshape(-1)
    H = np.zeros((6, 6), f32)
    habs = np.zeros(21)
    for q, (a, b) in enumerate(PAIRS):
        prod = sdf[a] * sdf[b]
        H[a, b] = H[b, a] = orc.esum(prod)
        habs[q] = np.abs(prod.astype(f64)).sum()
    jp = sdf * pdf
    jtr = np.array([orc.esum(jp[k]) for k in range(6)], f32)
    return dict(H=H, jtr=jtr, dp=orc.solve6(H, jtr), ssr=f32(orc.esum(pdf * pdf)), nvis=nvis, pt_ssr=pt_ssr,
                habs=habs, jabs=np.abs(jp.astype(f64)).sum(1), ssr_d=float((pdf.astype(f64) ** 2).sum()))


def evaluate_batch(orc, op, fc, cc, wh, planes_I, planes_dx, planes_dy, pt_off, pts, ref_frame, new_frame, p_ref,
                   p_cur=None, level=None):
    """A batch over flat per-frame plane sets (one per frame, laid out as ict_pyramid_layout); pt_ssr laid out like the
    points.  level defaults to lv_l."""
    level = op.lv_l if level is None else level
    cam = orc.camera_levels(op.lv_f + 1, fc, cc, wh, op.psz)
    _, offs, sw, _ = O.pyramid_layout(int(wh[0]), int(wh[1]), op.lv_f, op.psz)
    keys = ("H", "jtr", "dp", "ssr", "nvis", "habs", "jabs", "ssr_d")
    out = {k: [] for k in keys}
    pt_ssr = []
    for t in range(len(pt_off) - 1):
        a, b = int(pt_off[t]), int(pt_off[t + 1])
        rf, nf = int(ref_frame[t]), int(new_frame[t])
        r = evaluate_track(orc, op, cam, (planes_I[rf], planes_dx[rf], planes_dy[rf]), (planes_I[nf],), offs, sw,
                           np.asarray(pts[3 * a:3 * b], f64), p_ref[t], None if p_cur is None else p_cur[t], level)
        for k in keys:
            out[k].append(r[k])
        pt_ssr.append(r["pt_ssr"])
    res = {k: np.array(v) for k, v in out.items()}
    res["ssr"] = res["ssr"].astype(f32)
    res["nvis"] = res["nvis"].astype(np.int32)
    res["pt_ssr"] = np.concatenate(pt_ssr) if pt_ssr else np.zeros(0, f32)
    return res
