"""Cost of ict_track_evaluate against ict_track_batch on the same batch, in sum orders 1 (reference) and 0 (fast):

  psz32    4096 four-point 32x32 tracks on one 1080p pair (bench.py's geometry, BASELINE configs[2])
  psz8     256 hundred-point 8x8 tracks on one 640x480 pair (the template of BASELINE configs[1])
  dense    1080p, one point per pixel, psz 1 (BASELINE configs[3])

evaluate measures at level lv_l with p_cur = the tracked pose and no per-point output.  Times are host wall clock
around blocking calls (each ends in a device synchronise: small host<->device copies included), best and median of
REPS after one warm-up call.  Prints one JSON object with the card's name and power limit.

    python profiles/tools/evaluate_time.py [--reps 5] [--out FILE]
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


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return dict(best_ms=1e3 * min(ts), median_ms=1e3 * float(np.median(ts)))


def workload(name, w, h, psz, pt_off, pts, reps, seed):
    sc, A, B, _ = synth.make_pair(seed, w, h)
    fr = ict.Frames(2, w, h, 3, psz)
    fr.upload(0, np.stack([A, B]))
    T = len(pt_off) - 1
    op = ict.make_optparam(lv_f=3, lv_l=0, psz=psz, maxiter=10, normdp_ratio=0.01, maxpttrack=int(np.diff(pt_off).max()))
    res = {}
    for order in (1, 0):
        tr = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
        tr.set_sum_order(order)
        tr.set_points(pt_off, pts(sc).copy())
        p0 = np.zeros((T, 6))
        p = tr.track_batch(fr, 0, 1, p0)["p_out"]
        tb = timed(lambda: tr.track_batch(fr, 0, 1, p0), reps)
        ev = timed(lambda: tr.evaluate(fr, 0, 1, p0, p, 0), reps)
        res["order%d" % order] = dict(track_batch=tb, evaluate=ev,
                                      evaluate_over_track_batch=ev["median_ms"] / tb["median_ms"])
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
        "psz32", 1920, 1080, 32, np.arange(T + 1, dtype=np.int64) * 4,
        lambda sc: np.concatenate([sc.points(7000 + t, 4, 32, 3) for t in range(T)]), a.reps, 91)
    S = 256
    out["psz8_256x100_640x480"] = workload(
        "psz8", 640, 480, 8, np.arange(S + 1, dtype=np.int64) * 100,
        lambda sc: np.concatenate([sc.points(100 + s, 100, 8, 3) for s in range(S)]), a.reps, 5)
    sc_d, _, _, _ = synth.make_pair(3, 1920, 1080)
    n = sc_d.dense_points(16).size // 3
    out["dense_1080p"] = workload("dense", 1920, 1080, 1, np.array([0, n], np.int64), lambda sc: sc.dense_points(16),
                                  a.reps, 3)
    out["dense_1080p"]["points"] = n
    s = json.dumps(out, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s)


if __name__ == "__main__":
    main()
