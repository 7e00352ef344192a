#!/usr/bin/env python
"""Generates the golden fixtures in this directory.  Run in the BUILD container only (needs /root/reference for
oracle/_ref and Python cv2):   python tests/golden/make_golden.py

  pyramid_*.npz   util_constructpyramide computed with Python cv2 (an independent implementation of the three OpenCV
                  calls at utilities.cpp:24,30-31,40-46) on uint8-valued images.
  track_*.npz     inputs and outputs of the reference's OWN sources (oracle/_ref: utilities/camera/pose/odometer.cpp
                  compiled against oracle/shim) for Set3Dpoints -> SetPose -> TrackPose, with the per-iteration
                  (H, J^T r, delta_p) recorded by the shim's fullPivLu().solve() hook.
  se3.npz         util_SE3_coeff_to_group / util_SE3_group_to_coeff, float and double instantiations (oracle/_ref).
  getpatch.npz    util_getPatch / util_getPatch_grad at awkward centres (integers >= 256, frac > 1-1e-5, odd psz).
  drivers_stale.npz  run_track_nposes.cpp on a pan in which border points leave the frames mid-chain: pins the state
                  the reference keeps BETWEEN TrackPose calls (ResetOdometer only runs from Set3Dpoints).
  drivers.npz     inputs and outputs of the reference's own main()s: run_track_nposes.cpp (text in/out, forward and
                  backward chains, NCC) and run_io_reprojection_test.cpp (binary in/out), compiled into oracle/_ref.
  vs_ref.npz      what tests/test_oracle_vs_ref.py compares with: pyramids (digest + sample), traces, poses,
                  reprojections and centred points of its seeded cases, camera levels and one batch.  This script
                  records it from oracle/_ref.  The committed file holds the ORACLE's outputs instead: the reference's
                  sources were not at hand when it was recorded (see that test's docstring).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import oracle as O          # noqa: E402
from invcompcamtrack_b200 import synth  # noqa: E402


def cv2_pyramid(img_u8, lv_f, pad):
    import cv2
    prev = img_u8.astype(np.float32)
    I, dx, dy = [], [], []
    for l in range(lv_f + 1):
        cur = prev.copy() if l == 0 else cv2.resize(prev, None, fx=.5, fy=.5, interpolation=cv2.INTER_LINEAR)
        gx = cv2.Sobel(cur, cv2.CV_32F, 1, 0, ksize=1, scale=1, delta=0, borderType=cv2.BORDER_DEFAULT)
        gy = cv2.Sobel(cur, cv2.CV_32F, 0, 1, ksize=1, scale=1, delta=0, borderType=cv2.BORDER_DEFAULT)
        I.append(cv2.copyMakeBorder(cur, pad, pad, pad, pad, cv2.BORDER_REPLICATE).reshape(-1))
        dx.append(cv2.copyMakeBorder(gx, pad, pad, pad, pad, cv2.BORDER_CONSTANT, value=0).reshape(-1))
        dy.append(cv2.copyMakeBorder(gy, pad, pad, pad, pad, cv2.BORDER_CONSTANT, value=0).reshape(-1))
        prev = cur
    return np.concatenate(I), np.concatenate(dx), np.concatenate(dy)


def gen_pyramids():
    rng = np.random.default_rng(11)
    cases = {"rand": (rng.integers(0, 256, (64, 96)).astype(np.uint8), 3, 5),
             "sqrt": (synth.sqrt_image(160, 120), 2, 8),                      # run_io_test.m:8-14
             "tex": (synth.make_texture(5, 48, 64), 2, 1)}
    for name, (img, lv_f, pad) in cases.items():
        I, dx, dy = cv2_pyramid(img, lv_f, pad)
        np.savez_compressed(os.path.join(HERE, "pyramid_%s.npz" % name), img=img, lv_f=lv_f, pad=pad, I=I, dx=dx, dy=dy)


TRACK_CASES = {
    "base": dict(seed=3, w=160, h=120, psz=8, npts=40, lv_f=2),
    "donorm": dict(seed=4, w=160, h=120, psz=8, npts=40, lv_f=2, donorm=1),
    "patchnorm": dict(seed=5, w=160, h=120, psz=8, npts=40, lv_f=2, dopatchnorm=1),
    "both_odd": dict(seed=6, w=160, h=120, psz=5, npts=30, lv_f=1, donorm=1, dopatchnorm=1),
    "stale": dict(seed=7, w=160, h=120, psz=8, npts=40, lv_f=2, scale=6.0, edge=True),   # points leave the frames
    "psz4_cap": dict(seed=8, w=160, h=120, psz=4, npts=50, lv_f=2, maxpttrack=32),
}


def build_track_inputs(kw):
    kw = dict(kw)
    edge = kw.pop("edge", False)
    seed, w, h = kw.pop("seed"), kw.pop("w"), kw.pop("h")
    scale = kw.pop("scale", 1.0)
    npts = kw.pop("npts")
    sc, A, B, p_gt = synth.make_pair(seed, w, h, motion_scale=scale)
    if edge:   # put the points near the border so that some fall outside at some levels / iterations
        rng = np.random.default_rng(seed)
        u = np.concatenate([rng.uniform(0, 6, npts // 2), rng.uniform(w - 8, w - 0.5, npts - npts // 2)])
        v = rng.uniform(1, h - 1, npts)
        d = np.stack([(u - sc.cc[0]) / sc.fc[0], (v - sc.cc[1]) / sc.fc[1], np.ones(npts)], 0) * sc.depth
        pts = np.ascontiguousarray(d.reshape(-1), np.float64)
    else:
        pts = sc.points(seed, npts, kw["psz"], kw["lv_f"])
    op = O.make_optparam(maxpttrack=kw.pop("maxpttrack", npts), **kw)
    return sc, A, B, p_gt, pts, op


def gen_tracks(ref):
    for name, kw in TRACK_CASES.items():
        sc, A, B, p_gt, pts, op = build_track_inputs(kw)
        lv_f, psz = op.lv_f, op.psz
        tot, off, sw, sh = O.pyramid_layout(A.shape[1], A.shape[0], lv_f, psz)
        pa = ref.pyramid_build(A.astype(np.float32), lv_f, psz)
        pb = ref.pyramid_build(B.astype(np.float32), lv_f, psz)
        od = O.Odometer(ref, op, sc.fc, sc.cc, sc.wh)
        pmut = pts.copy()
        od.set3dpoints(pmut)
        p_in = np.zeros(6) if name != "donorm" else np.array([0.01, -0.02, 0.005, 0.002, -0.001, 0.003])
        od.setpose(p_in, pa, pb, lv_f, off)
        pt2d = od.get2dpoints()
        p_out, solves = ref.track(od, 128)
        od.close()
        np.savez_compressed(os.path.join(HERE, "track_%s.npz" % name), A=A, B=B, pts=pts, pts_after=pmut, p_in=p_in,
                            fc=sc.fc, cc=sc.cc, wh=sc.wh, op=np.frombuffer(bytes(op), np.uint8), p_out=p_out,
                            solves=solves, pt2d=pt2d, p_gt=p_gt)
        print(name, "iterations", len(solves), "p_out", p_out)


def gen_se3(ref):
    rng = np.random.default_rng(2)
    P = np.concatenate([rng.uniform(-1, 1, (24, 6)) * np.array([1, 1, 1, .5, .5, .5]),
                        rng.uniform(-1, 1, (8, 6)) * np.array([1, 1, 1, 2e-5, 2e-5, 2e-5]),    # Taylor branch
                        np.zeros((1, 6))])
    Gf = np.stack([ref.se3_exp(p, np.float32) for p in P])
    Gd = np.stack([ref.se3_exp(p, np.float64) for p in P])
    Gf_full, Gd_full = Gf.copy(), Gd.copy()
    lf = np.stack([ref.se3_log(g, np.float32) for g in Gf_full])
    ld = np.stack([ref.se3_log(g, np.float64) for g in Gd_full])
    np.savez_compressed(os.path.join(HERE, "se3.npz"), P=P, Gf=Gf, Gd=Gd, lf=lf, ld=ld)


def gen_getpatch(ref):
    rng = np.random.default_rng(9)
    w, h, pad = 640, 64, 8
    img = rng.integers(0, 256, (h, w)).astype(np.float32)
    out = {}
    for psz in (8, 5, 1):
        I, dx, dy = ref.pyramid_build(img, 0, psz)
        width = w + 2 * psz
        mids = np.array([[5.0, 7.0], [255.0, 10.0], [256.0, 10.0], [300.0, 20.0], [512.0, 33.0], [100.25, 40.75],
                         [17.999995, 12.5], [300.99999, 9.000001], [0.0, 0.0], [float(w), float(h)], [639.5, 63.5]],
                        np.float32)
        for pn in (0, 1):
            op = O.make_optparam(lv_f=0, psz=psz, dopatchnorm=pn, maxpttrack=4)
            pat = np.stack([ref.getpatch(I, m, op, width) for m in mids])
            g = [ref.getpatch_grad(I, dx, dy, m, op, width) for m in mids]
            out["p%d_n%d" % (psz, pn)] = pat
            out["g%d_n%d" % (psz, pn)] = np.stack([np.stack(x) for x in g])
        out["mids"] = mids
    np.savez_compressed(os.path.join(HERE, "getpatch.npz"), img=img, **out)


def write_pgm(path, img):
    with open(path, "wb") as f:
        f.write(b"P5\n%d %d\n255\n" % (img.shape[1], img.shape[0]))
        f.write(np.ascontiguousarray(img, np.uint8).tobytes())


def nposes_inputs():
    """A small run_track_nposes problem: 4 frames (1 back, 2 forward), 60 correspondences, 3 pose samples."""
    sc, frames, poses = synth.make_sequence(9, 4, 160, 120, motion_scale=0.3)
    nb, nf = 1, 2
    pts = sc.points(5, 60, 8, 2, p_ref=poses[nb]).reshape(3, -1).T          # world points seen in the reference frame
    rng = np.random.default_rng(4)
    samples = []
    for s in range(3):
        p = poses[nb] + rng.normal(0, 1, 6) * np.array([2e-3, 2e-3, 2e-3, 3e-4, 3e-4, 3e-4]) * (s > 0)
        ids = np.sort(rng.choice(60, size=(24, 32, 40)[s], replace=False)) + 1
        samples.append((p, ids))
    lines = ["2 0 8 10 0.01 0 0 40 0", "%g %g %g %g %d %d" % (sc.fc[0], sc.fc[1], sc.cc[0], sc.cc[1], 160, 120),
             "%d %d" % (nb, nf)]
    lines += ["@DIR@/f%d.pgm" % k for k in range(4)]
    lines.append("%d" % len(pts))
    lines += ["0 0 %.17g %.17g %.17g" % tuple(x) for x in pts]
    lines.append("%d" % len(samples))
    for p, ids in samples:
        lines.append(" ".join("%.17g" % v for v in p) + " %d " % len(ids) + " ".join(str(i) for i in ids))
    return frames, "\n".join(lines) + "\n", sc


def nposes_stale_inputs():
    """run_track_nposes with points that LEAVE the frames mid-chain (SURVEY.md §8 a4: state between TrackPose calls): a
    sideways pan over 6 frames (2 back, 3 forward of the reference frame), half of the correspondences within 12 px of
    the left / right border of the reference frame, 4 pose samples."""
    w, h, nb, nf = 160, 120, 2, 3
    sc = synth.Scene(19, w, h)
    nfr = nb + nf + 1
    poses = np.zeros((nfr, 6))
    for k in range(nfr):                       # pan: ~7 px per frame at level 0, plus a little roll
        poses[k] = np.array([0.22 * (k - nb), 0.02 * (k - nb), 0.0, 0.0, 0.0, 0.004 * (k - nb)])
    frames = [sc.render(poses[k]) for k in range(nfr)]
    rng = np.random.default_rng(14)
    n = 64
    u = np.concatenate([rng.uniform(1, 12, n // 4), rng.uniform(w - 12, w - 1, n // 4), rng.uniform(20, w - 20, n // 2)])
    v = rng.uniform(10, h - 10, n)
    pts = sc.backproject(u, v, poses[nb]).reshape(3, -1).T
    samples = []
    for s_ in range(4):
        p = poses[nb] + rng.normal(0, 1, 6) * np.array([2e-3, 2e-3, 2e-3, 3e-4, 3e-4, 3e-4]) * (s_ > 0)
        ids = np.sort(rng.choice(n, size=(40, 48, 36, 44)[s_], replace=False)) + 1
        samples.append((p, ids))
    lines = ["2 0 8 10 0.01 0 0 48 0", "%g %g %g %g %d %d" % (sc.fc[0], sc.fc[1], sc.cc[0], sc.cc[1], w, h),
             "%d %d" % (nb, nf)]
    lines += ["@DIR@/f%d.pgm" % k for k in range(nfr)]
    lines.append("%d" % len(pts))
    lines += ["0 0 %.17g %.17g %.17g" % tuple(x) for x in pts]
    lines.append("%d" % len(samples))
    for p, ids in samples:
        lines.append(" ".join("%.17g" % v_ for v_ in p) + " %d " % len(ids) + " ".join(str(i) for i in ids))
    return frames, "\n".join(lines) + "\n"


def gen_drivers_stale():
    import subprocess
    import tempfile
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    frames, template = nposes_stale_inputs()
    with tempfile.TemporaryDirectory() as d:
        for k, f in enumerate(frames):
            write_pgm(os.path.join(d, "f%d.pgm" % k), f)
        open(os.path.join(d, "in.txt"), "w").write(template.replace("@DIR@", d))
        subprocess.run([os.path.join(ref_dir, "run_track_nposes"), os.path.join(d, "in.txt"), os.path.join(d, "out.txt")],
                       check=True)
        out = open(os.path.join(d, "out.txt")).read()
    np.savez_compressed(os.path.join(HERE, "drivers_stale.npz"), frames=np.stack(frames), nposes_input=template,
                        nposes_output=out)
    print("run_track_nposes (points leaving the frames) golden:\n" + out[:600])


def gen_drivers():
    """Golden outputs of the reference's own DRIVERS (oracle/_ref/run_track_nposes, run_io_reprojection_test: the
    reference mains compiled against the stand-in headers; the stand-in imread reads binary PGM)."""
    import struct
    import subprocess
    import tempfile
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    frames, template, sc = nposes_inputs()
    with tempfile.TemporaryDirectory() as d:
        for k, f in enumerate(frames):
            write_pgm(os.path.join(d, "f%d.pgm" % k), f)
        open(os.path.join(d, "in.txt"), "w").write(template.replace("@DIR@", d))
        subprocess.run([os.path.join(ref_dir, "run_track_nposes"), os.path.join(d, "in.txt"), os.path.join(d, "out.txt")],
                       check=True)
        out = open(os.path.join(d, "out.txt")).read()
        # single pair: frames 1 -> 2, 50 points, binary input of run_io_reprojection_test.cpp:54-79
        pts = sc.points(6, 50, 8, 2).reshape(3, -1)
        blob = struct.pack("<6d2f2f2IQ", *([0.0] * 6), float(sc.fc[0]), float(sc.fc[1]), float(sc.cc[0]), float(sc.cc[1]),
                           160, 120, 50)
        blob += pts.astype("<f8").tobytes() + np.zeros(100, "<f4").tobytes()
        open(os.path.join(d, "pair.bin"), "wb").write(blob)
        args = "2 0 8 10 0.01 0 0 50 0".split()
        subprocess.run([os.path.join(ref_dir, "run_io_reprojection_test"), os.path.join(d, "f0.pgm"),
                        os.path.join(d, "f1.pgm"), os.path.join(d, "pair.bin"), os.path.join(d, "pair.out")] + args,
                       check=True)
        pair_out = np.frombuffer(open(os.path.join(d, "pair.out"), "rb").read(), "<f8")
    np.savez_compressed(os.path.join(HERE, "drivers.npz"), frames=np.stack(frames), nposes_input=template,
                        nposes_output=out, pair_input=np.frombuffer(blob, np.uint8), pair_args=" ".join(args),
                        pair_output=pair_out)
    print("run_track_nposes golden:\n" + out[:400])
    print("run_io_reprojection_test golden:", pair_out)


def gen_vs_ref(ref):
    """Records from the reference only: an oracle recording would pin the oracle to itself."""
    assert isinstance(ref, O.RefLib)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import ref_outputs
    np.savez_compressed(os.path.join(HERE, "vs_ref.npz"), **ref_outputs(ref, O.OracleLib()))


if __name__ == "__main__":
    O.build("ref")
    ref = O.RefLib()
    gen_pyramids()
    gen_tracks(ref)
    gen_se3(ref)
    gen_getpatch(ref)
    gen_drivers()
    gen_drivers_stale()
    gen_vs_ref(ref)
    print("golden fixtures written to", HERE)
