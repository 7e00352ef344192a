"""CPU: pins the CPU model of ict_track_evaluate (tests/evaluate_model.py) to the oracle's TrackPose.

  * at the SetPose pose and level lv_f it reproduces TrackPose's first iteration (J^T r, delta_p, visible points) bit
    for bit, in sum modes 0 and 1, on tracks of every shape;
  * with donorm = 0, at the pose TrackPose holds when it enters level l, it reproduces the first iteration of that level
    at every level, and its Hessian at lv_l is TrackPose's;
  * its SSR and per-point sums agree with a float64 sum of (template - new patch)^2 built from getpatch_grad / getpatch.
"""
import numpy as np
import pytest

from oracle import oracle as O
from helpers import make_case
from evaluate_model import evaluate_track, evaluate_batch

# (case options, initial pose): odd psz, dopatchnorm, donorm, a maxpttrack cap, points near the border that leave the
# new frame, large motion
CASES = [
    (dict(seed=201, psz=8, npts=40, lv_f=3, dopatchnorm=1), None),
    (dict(seed=202, psz=4, npts=50, lv_f=2, maxpttrack=32), None),
    (dict(seed=203, psz=7, npts=30, lv_f=2, dopatchnorm=1), None),
    (dict(seed=204, psz=5, npts=30, lv_f=1, donorm=1, dopatchnorm=1), [0.01, -0.02, 0.005, 0.002, -0.001, 0.003]),
    (dict(seed=205, psz=8, npts=40, lv_f=2, scale=4.0), [1.2, 0.3, 0.0, 0.0, 0.02, 0.0]),
]


def pyramids(orc, c):
    return (orc.pyramid_build(c["A"].astype(np.float32), c["lv_f"], c["psz"]),
            orc.pyramid_build(c["B"].astype(np.float32), c["lv_f"], c["psz"]))


def odometer(orc, c, pa, pb, p_in, pts=None):
    _, offs, _, _ = O.pyramid_layout(c["w"], c["h"], c["lv_f"], c["psz"])
    od = O.Odometer(orc, c["op"], c["sc"].fc, c["sc"].cc, c["sc"].wh)
    od.set3dpoints((c["pts"] if pts is None else pts).copy())
    od.setpose(p_in, pa, pb, c["lv_f"], offs)
    return od


def model(orc, c, pa, pb, p_ref, level, p_cur=None):
    op = c["op"]
    _, offs, sw, _ = O.pyramid_layout(c["w"], c["h"], c["lv_f"], c["psz"])
    cam = orc.camera_levels(op.lv_f + 1, c["sc"].fc, c["sc"].cc, c["sc"].wh, op.psz)
    return evaluate_track(orc, op, cam, pa, pb, offs, sw, c["pts"], p_ref, p_cur, level)


def case_of(kw, p):
    c = make_case(**kw)
    return c, np.zeros(6) if p is None else np.asarray(p, np.float64)


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("k", range(len(CASES)))
def test_first_iteration(orc, k, mode):
    c, p_in = case_of(*CASES[k])
    pa, pb = pyramids(orc, c)
    orc.set_sum_mode(mode)
    try:
        e = model(orc, c, pa, pb, p_in, c["lv_f"])
        od = odometer(orc, c, pa, pb, p_in)
        _, _, tr, _ = orc.track(od, 64)
        od.close()
    finally:
        orc.set_sum_mode(0)
    assert np.array_equal(e["jtr"], tr[0, 2:8])
    assert np.array_equal(e["dp"], tr[0, 8:14])
    assert e["nvis"] == tr[0, 15]


def entry_poses(trace, p_in):
    """The fp32 pose TrackPose holds when it enters each level: float32(p_in) + the running fp32 sum of delta_p."""
    p = np.asarray(p_in, np.float64).astype(np.float32)
    out = {}
    for r in trace:
        lv = int(r[0])
        if lv not in out:
            out[lv] = p.copy()
        p = (p + r[8:14].astype(np.float32)).astype(np.float32)
    return out


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("k", [0, 1, 2, 4])    # donorm = 0
def test_every_level_and_hessian(orc, k, mode):
    c, p_in = case_of(*CASES[k])
    pa, pb = pyramids(orc, c)
    orc.set_sum_mode(mode)
    try:
        od = odometer(orc, c, pa, pb, p_in)
        _, _, tr, _ = orc.track(od, 96)
        H_last = orc.hessian(od)
        first = {}
        for r in tr:
            first.setdefault(int(r[0]), r)
        for lv, p in entry_poses(tr, p_in).items():
            e = model(orc, c, pa, pb, p_in, lv, p.astype(np.float64))
            assert np.array_equal(e["jtr"], first[lv][2:8]), lv
            assert np.array_equal(e["dp"], first[lv][8:14]), lv
            assert e["nvis"] == first[lv][15], lv
        e = model(orc, c, pa, pb, p_in, c["op"].lv_l)
        assert np.array_equal(e["H"], H_last)
        od.close()
    finally:
        orc.set_sum_mode(0)


def test_uneven_and_empty_tracks(orc):
    """A batch with tracks of 0, 1, 37 and 5 points and a capped one: the batch evaluation equals each track's first
    trace record; pt_ssr is -1 beyond maxpttrack."""
    c = make_case(seed=206, psz=8, npts=60, lv_f=2, maxpttrack=40)
    pa, pb = pyramids(orc, c)
    sizes = [5, 0, 1, 37, 60]
    pts = [c["sc"].points(900 + t, n, 8, 2) for t, n in enumerate(sizes)]
    pt_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    allp = np.concatenate(pts)
    T = len(sizes)
    p_in = np.zeros((T, 6)); p_in[2, 0] = 0.05
    planes = [[pa[q], pb[q]] for q in range(3)]
    rf, nf = np.zeros(T, np.int32), np.ones(T, np.int32)
    o = orc.track_batch(c["op"], c["sc"].fc, c["sc"].cc, c["sc"].wh, *planes, pt_off, allp.copy(), rf, nf, p_in,
                        trace_cap=64, nthreads=1)
    e = evaluate_batch(orc, c["op"], c["sc"].fc, c["sc"].cc, c["sc"].wh, *planes, pt_off, allp, rf, nf, p_in,
                       level=c["lv_f"])
    assert np.array_equal(e["jtr"], o["trace"][:, 0, 2:8])
    assert np.array_equal(e["dp"], o["trace"][:, 0, 8:14])
    assert np.array_equal(e["nvis"], o["trace"][:, 0, 15])
    assert (e["H"][1] == 0).all() and e["ssr"][1] == 0
    assert (e["pt_ssr"][pt_off[4] + 40:] == -1).all() and (e["pt_ssr"][pt_off[4]:pt_off[4] + 40] >= 0).any()


def project(G, X, Y, Z, cam, l):
    """project_pt in fp32, the reference's association."""
    f = np.float32
    tx = G[0] * X + G[1] * Y + G[2] * Z + G[3]
    ty = G[4] * X + G[5] * Y + G[6] * Z + G[7]
    tz = G[8] * X + G[9] * Y + G[10] * Z + G[11]
    return (tx / tz) * f(cam[l, 0]) + f(cam[l, 2]), (ty / tz) * f(cam[l, 1]) + f(cam[l, 3])


def inside(x, y, cam, l):
    return bool((x >= 0) & (y >= 0) & (x <= cam[l, 4]) & (y <= cam[l, 5]))


@pytest.mark.parametrize("k", [0, 2, 4])
def test_ssr_against_float64_patches(orc, k):
    """sum (template - new patch)^2 in float64 from getpatch_grad / getpatch, the template taken at the finest level in
    [level, lv_f] where the point is inside the reference image."""
    c, p_in = case_of(*CASES[k])
    pa, pb = pyramids(orc, c)
    op = c["op"]
    _, offs, sw, _ = O.pyramid_layout(c["w"], c["h"], c["lv_f"], c["psz"])
    cam = orc.camera_levels(op.lv_f + 1, c["sc"].fc, c["sc"].cc, c["sc"].wh, op.psz)
    n = c["pts"].size // 3
    P = min(n, op.maxpttrack)
    X, Y, Z = (c["pts"][j * n:(j + 1) * n].astype(np.float32) for j in range(3))
    p_cur = p_in + np.array([0.002, -0.001, 0.0, 0.0005, 0.0, -0.0003])
    Gr = orc.se3_exp(p_in.astype(np.float32))
    Gc = orc.se3_exp(p_cur.astype(np.float32))
    plane = lambda a, l: a[offs[l]:]          # noqa: E731
    for level in range(op.lv_l, op.lv_f + 1):
        e = model(orc, c, pa, pb, p_in, level, p_cur)
        tot = 0.0
        for i in range(P):
            tmpl = np.zeros(op.novals, np.float32)
            for l in range(op.lv_f, level - 1, -1):
                x, y = project(Gr, X[i], Y[i], Z[i], cam, l)
                if inside(x, y, cam, l):
                    tmpl = orc.getpatch_grad(plane(pa[0], l), plane(pa[1], l), plane(pa[2], l), [x, y], op, sw[l])[0]
            x, y = project(Gc, X[i], Y[i], Z[i], cam, level)
            if not inside(x, y, cam, level):
                assert e["pt_ssr"][i] == -1
                continue
            new = orc.getpatch(plane(pb[0], level), [x, y], op, sw[level])
            s = float(((tmpl.astype(np.float64) - new.astype(np.float64)) ** 2).sum())
            assert abs(e["pt_ssr"][i] - s) <= 1e-6 * max(s, 1e-30), (level, i, e["pt_ssr"][i], s)
            tot += s
        assert abs(e["ssr"] - tot) <= 1e-6 * tot, (level, e["ssr"], tot)
        assert abs(e["ssr_d"] - tot) <= 1e-6 * tot


def test_reference_visibility_is_level_independent(orc):
    """The per-level intrinsics are exact powers-of-two scalings (camera.cpp:34) and so is every projected coordinate,
    so a point inside the reference image at one level is inside at all: within one SetPose no template slot goes stale
    (the walk over the levels still follows TrackPose).  Border points of a case built for it confirm this."""
    c, p_in = case_of(*CASES[4])
    op = c["op"]
    cam = orc.camera_levels(op.lv_f + 1, c["sc"].fc, c["sc"].cc, c["sc"].wh, op.psz)
    rng = np.random.default_rng(7)
    u = np.concatenate([rng.uniform(-0.5, 0.5, 200), c["w"] + rng.uniform(-0.5, 0.5, 200)])
    v = rng.uniform(1, c["h"] - 1, 400)
    X = ((u - c["sc"].cc[0]) / c["sc"].fc[0] * 5).astype(np.float32)
    Y = ((v - c["sc"].cc[1]) / c["sc"].fc[1] * 5).astype(np.float32)
    Z = np.full(400, 5, np.float32)
    G = orc.se3_exp(np.zeros(6, np.float32))
    for i in range(400):
        vis = {inside(*project(G, X[i], Y[i], Z[i], cam, l), cam, l) for l in range(op.lv_f + 1)}
        assert len(vis) == 1, i
