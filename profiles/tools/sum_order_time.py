"""Reference summation order with Eigen's 4-float SSE packets (sum order 1, eight chains per sum) against 8-float AVX
packets (sum order 3, sixteen chains), on four workloads, with the two orders alternated in one process:

  configs[0]   one 100-point 8x8 track, 640x480 (bench.py other_configs.single_pair)      K2x8
  configs[1]   256 chains of one 100-point 8x8 template over 100 frames (chain_100_frames)  K2x8
  psz32        8192 four-point 32x32 tracks on one 1080p pair                              order 1: K2r, order 3: k_track
  dense        1080p, one point per pixel, psz 1 (dense_1080p)                              multi-CTA path

Times are host wall clock around blocking calls (each ends in a device synchronise), best and median of REPS after one
warm-up call.  On a sample of each workload order 3 is compared with the oracle in its sum mode 1 (order 1 with its
sum mode 0): poses, iteration counts and pixel-residual counts must be equal.  Prints one JSON object.

    python profiles/tools/sum_order_time.py [--reps 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

R = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, R)
import numpy as np  # noqa: E402

import invcompcamtrack_b200 as ict  # noqa: E402
from invcompcamtrack_b200 import synth  # noqa: E402
from oracle import oracle as O  # noqa: E402

ORACLE_MODE = {1: 0, 3: 1}      # library sum order -> oracle sum mode


def compare(orders, reps, make_run):
    """make_run(order) -> callable; orders alternate rep by rep so that both see the same machine state."""
    res = {o: [] for o in orders}
    outs = {}
    runs = {o: make_run(o) for o in orders}
    for o in orders:
        runs[o]()
    for _ in range(reps):
        for o in orders:
            t0 = time.perf_counter()
            outs[o] = runs[o]()
            res[o].append(time.perf_counter() - t0)
    return {o: dict(best_ms=1e3 * min(v), median_ms=1e3 * float(np.median(v))) for o, v in res.items()}, outs


def same(g, o, keys=("p_out", "iters", "npixres")):
    return all(np.array_equal(np.asarray(g[k]), np.asarray(o[k])) for k in keys)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    dev = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        dev["power_limit_and_max_sm_clock"] = q[0] if q else None
    except (OSError, subprocess.SubprocessError):
        dev["power_limit_and_max_sm_clock"] = None
    orc = O.OracleLib()
    orders = (1, 3)
    out = {"device": dev, "reps": a.reps, "timing": "host wall clock around blocking calls, after one warm-up call"}

    def oracle_batch(op_o, sc, pyr, pt_off, pts, ref, new, p_in, order):
        orc.set_sum_mode(ORACLE_MODE[order])
        try:
            return orc.track_batch(op_o, sc.fc, sc.cc, sc.wh, [q[0] for q in pyr], [q[1] for q in pyr],
                                   [q[2] for q in pyr], pt_off, pts.copy(), ref, new, p_in, nthreads=os.cpu_count() or 1)
        finally:
            orc.set_sum_mode(0)

    # ---- configs[0] ---------------------------------------------------------------------------------------------------
    sc, A, B, _ = synth.make_pair(7, 640, 480)
    pts = sc.points(911, 100, 8, 3)
    kw = dict(lv_f=3, lv_l=0, psz=8, maxiter=10, normdp_ratio=0.01, donorm=0, dopatchnorm=0, maxpttrack=100)
    op, op_o = ict.make_optparam(**kw), O.make_optparam(**kw)
    fr = ict.Frames(2, 640, 480, 3, 8)
    fr.upload(0, np.stack([A, B]))
    trs = {}
    for o in orders:
        trs[o] = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
        trs[o].set_sum_order(o)
        trs[o].set_points(np.array([0, 100], np.int64), pts.copy())
    t, g = compare(orders, 4 * a.reps, lambda o: (lambda: trs[o].track_batch(fr, 0, 1, np.zeros((1, 6)))))
    pyr = [orc.pyramid_build(x.astype(np.float32), 3, 8) for x in (A, B)]
    out["configs0_single_pair"] = {
        o: dict(t[o], iters=int(g[o]["iters"].sum()), bit_identical_to_oracle=same(
            g[o], oracle_batch(op_o, sc, pyr, np.array([0, 100]), pts, [0], [1], np.zeros((1, 6)), o)))
        for o in orders}
    for o in orders:
        trs[o].close()
    fr.close()

    # ---- configs[1] ---------------------------------------------------------------------------------------------------
    NF, S = 100, 256
    sc, frames, _ = synth.make_sequence(5, NF, 640, 480)
    fr = ict.Frames(NF, 640, 480, 3, 8)
    fr.upload(0, np.stack(frames))
    cpts = np.concatenate([sc.points(100 + s_, 100, 8, 3) for s_ in range(S)])
    for o in orders:
        trs[o] = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
        trs[o].set_sum_order(o)
        trs[o].set_points(np.arange(S + 1, dtype=np.int64) * 100, cpts.copy())
    t, g = compare(orders, a.reps, lambda o: (lambda: trs[o].track_sequence(fr, 0, NF - 1, 1, np.zeros((S, 6)))))
    CS, CF = 8, 6                                # oracle sample: 8 chains over the first 6 frame steps
    pyr = [orc.pyramid_build(f.astype(np.float32), 3, 8) for f in frames[:CF + 1]]
    res = {}
    for o in orders:
        p, ok = np.zeros((CS, 6)), True
        for k in range(CF):
            r = oracle_batch(op_o, sc, pyr, np.arange(CS + 1, dtype=np.int64) * 100, cpts[:300 * CS],
                             np.full(CS, k, np.int32), np.full(CS, k + 1, np.int32), p, o)
            p = r["p_out"]
            ok &= np.array_equal(g[o]["poses"][k + 1, :CS], p) and np.array_equal(g[o]["iters"][k, :CS], r["iters"])
        res[o] = dict(t[o], pixel_residuals=int(g[o]["npixres"].sum()), bit_identical_on_sample=bool(ok),
                      sample="%d chains x %d frame steps" % (CS, CF))
    out["configs1_chain_100_frames"] = res
    for o in orders:
        trs[o].close()
    fr.close()

    # ---- 8192 four-point psz-32 tracks, 1080p -----------------------------------------------------------------------------
    T, P = 8192, 4
    sc, A, B, _ = synth.make_pair(91, 1920, 1080)
    pts = np.concatenate([sc.points(7000 + t_, P, 32, 3) for t_ in range(T)])
    kw = dict(lv_f=3, lv_l=0, psz=32, maxiter=10, normdp_ratio=0.01, donorm=0, dopatchnorm=0, maxpttrack=P)
    op, op_o = ict.make_optparam(**kw), O.make_optparam(**kw)
    fr = ict.Frames(2, 1920, 1080, 3, 32)
    fr.upload(0, np.stack([A, B]))
    for o in orders:
        trs[o] = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
        trs[o].set_sum_order(o)
        trs[o].set_points(np.arange(T + 1, dtype=np.int64) * P, pts.copy())
    t, g = compare(orders, a.reps, lambda o: (lambda: trs[o].track_batch(fr, 0, 1, np.zeros((T, 6)))))
    sub = np.arange(0, T, 128)
    pyr = [orc.pyramid_build(x.astype(np.float32), 3, 32) for x in (A, B)]
    spts = pts.reshape(T, 3 * P)[sub].reshape(-1)
    res = {}
    for o in orders:
        r = oracle_batch(op_o, sc, pyr, np.arange(len(sub) + 1, dtype=np.int64) * P, spts, np.zeros(len(sub), np.int32),
                         np.ones(len(sub), np.int32), np.zeros((len(sub), 6)), o)
        gs = {k: g[o][k][sub] for k in ("p_out", "iters", "npixres")}
        npx = int(g[o]["npixres"].sum())
        res[o] = dict(t[o], pixel_residuals_per_s=npx / (1e-3 * t[o]["best_ms"]), bit_identical_on_sample=same(gs, r),
                      sample="%d of %d tracks" % (len(sub), T))
    out["psz32_8192x4"] = res
    for o in orders:
        trs[o].close()
    fr.close()

    # ---- dense 1080p ------------------------------------------------------------------------------------------------------
    w, h = 1920, 1080
    sc, A, B, _ = synth.make_pair(41, w, h, tilt=(0.05, -0.03))
    pts = sc.dense_points(16)
    n = pts.size // 3
    kw = dict(lv_f=3, lv_l=0, psz=1, maxiter=10, normdp_ratio=0.01, donorm=0, dopatchnorm=0, maxpttrack=n)
    op, op_o = ict.make_optparam(**kw), O.make_optparam(**kw)
    fr = ict.Frames(2, w, h, 3, 1)
    fr.upload(0, np.stack([A, B]))
    for o in orders:
        trs[o] = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
        trs[o].set_sum_order(o)
        trs[o].set_points(np.array([0, n], np.int64), pts.copy())
    t, g = compare(orders, a.reps, lambda o: (lambda: trs[o].track_batch(fr, 0, 1, np.zeros((1, 6)))))
    pyr = [orc.pyramid_build(x.astype(np.float32), 3, 1) for x in (A, B)]
    out["dense_1080p"] = {
        o: dict(t[o], points=n, iters=int(g[o]["iters"].sum()), bit_identical_to_oracle=same(
            g[o], oracle_batch(op_o, sc, pyr, np.array([0, n]), pts, [0], [1], np.zeros((1, 6)), o)))
        for o in orders}
    for o in orders:
        trs[o].close()
    fr.close()

    s = json.dumps(out, indent=1, default=str)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s)


if __name__ == "__main__":
    main()
