"""Cost of ict_track_evaluate_poses (K candidate poses per track) against two ways of getting the same numbers from
ict_track_evaluate, in sum orders 1 (reference) and 0 (fast), at levels lv_f and lv_l:

  replicated   set_points with every track's points K times, one evaluate of the T*K tracks
  separate     K evaluate calls on the T tracks, one per candidate

  psz32    4096 four-point 32x32 tracks on one 1080p pair (bench.py's geometry), K = 16 and 64
  psz8     256 hundred-point 8x8 tracks on one 640x480 pair, K = 16 and 64
  dense    1080p, one point per pixel, psz 1, K = 4

Candidates: the tracked pose plus uniform perturbations (+-0.02 translation, +-0.005 rad).  Each setting also times
evaluate_poses at K = 1 against evaluate at the same pose, the two calls alternating.  Times are host wall clock around
blocking calls (each ends in a device synchronise: small host<->device copies included), best and median of REPS
after one warm-up call.  Prints one JSON object with the card's name and power limit.

    python profiles/tools/evaluate_poses_time.py [--reps 5] [--out FILE]
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


def stats(ts):
    return dict(best_ms=1e3 * min(ts), median_ms=1e3 * float(np.median(ts)))


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return stats(ts)


def alternating(fa, fb, reps):
    """fa and fb in turn, one warm-up call each: (stats of fa, stats of fb)."""
    fa(); fb()
    ta, tb = [], []
    for _ in range(reps):
        for f, ts in ((fa, ta), (fb, tb)):
            t0 = time.perf_counter()
            f()
            ts.append(time.perf_counter() - t0)
    return stats(ta), stats(tb)


def workload(w, h, psz, pt_off, pts, Ks, reps, seed):
    sc, A, B, _ = synth.make_pair(seed, w, h)
    fr = ict.Frames(2, w, h, 3, psz)
    fr.upload(0, np.stack([A, B]))
    T = len(pt_off) - 1
    sizes = np.diff(pt_off)
    op = ict.make_optparam(lv_f=3, lv_l=0, psz=psz, maxiter=10, normdp_ratio=0.01, maxpttrack=int(sizes.max()))
    P = pts(sc).copy()
    res = {}
    for order in (1, 0):
        tr = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
        tr.set_sum_order(order)
        tr.set_points(pt_off, P)
        p0 = np.zeros((T, 6))
        p = tr.track_batch(fr, 0, 1, p0)["p_out"]
        for level in (op.lv_f, op.lv_l):
            r = {}
            one_poses, one_eval = alternating(lambda: tr.evaluate_poses(fr, 0, 1, p0, p[:, None], level),
                                              lambda: tr.evaluate(fr, 0, 1, p0, p, level), reps)
            r["K1"] = dict(evaluate_poses=one_poses, evaluate=one_eval)
            for K in Ks:
                rng = np.random.default_rng(K)
                cand = p[:, None, :] + np.concatenate([rng.uniform(-0.02, 0.02, (T, K, 3)),
                                                       rng.uniform(-0.005, 0.005, (T, K, 3))], 2)
                new = timed(lambda: tr.evaluate_poses(fr, 0, 1, p0, cand, level), reps)
                sep = timed(lambda: [tr.evaluate(fr, 0, 1, p0, np.ascontiguousarray(cand[:, k]), level)
                                     for k in range(K)], max(1, reps // 2))
                # replicated: track t's points K times, tracks t*K + k
                rep = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
                rep.set_sum_order(order)
                segs = [P[3 * pt_off[t]:3 * pt_off[t + 1]] for t in range(T)]
                rep.set_points(np.concatenate([[0], np.cumsum(np.repeat(sizes, K))]).astype(np.int64),
                               np.concatenate([s for s in segs for _ in range(K)]))
                p0r, candr = np.repeat(p0, K, 0), cand.reshape(T * K, 6)
                repl = timed(lambda: rep.evaluate(fr, 0, 1, p0r, candr, level), max(1, reps // 2))
                rep.close()
                r["K%d" % K] = dict(evaluate_poses=new, replicated=repl, separate=sep,
                                    replicated_over_poses=repl["median_ms"] / new["median_ms"],
                                    separate_over_poses=sep["median_ms"] / new["median_ms"])
            res["order%d_level%d" % (order, level)] = r
        tr.close()
    fr.close()
    return res


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
    out = {"device": dev, "reps": a.reps, "timing": "host wall clock around blocking calls, after one warm-up call"}
    T = 4096
    out["psz32_4096x4_1080p"] = workload(
        1920, 1080, 32, np.arange(T + 1, dtype=np.int64) * 4,
        lambda sc: np.concatenate([sc.points(7000 + t, 4, 32, 3) for t in range(T)]), (16, 64), a.reps, 91)
    S = 256
    out["psz8_256x100_640x480"] = workload(
        640, 480, 8, np.arange(S + 1, dtype=np.int64) * 100,
        lambda sc: np.concatenate([sc.points(100 + s, 100, 8, 3) for s in range(S)]), (16, 64), a.reps, 5)
    sc_d, _, _, _ = synth.make_pair(3, 1920, 1080)
    n = sc_d.dense_points(16).size // 3
    out["dense_1080p"] = workload(1920, 1080, 1, np.array([0, n], np.int64), lambda sc: sc.dense_points(16), (4,),
                                  max(1, a.reps // 2), 3)
    out["dense_1080p"]["points"] = n
    s = json.dumps(out, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s)


if __name__ == "__main__":
    main()
