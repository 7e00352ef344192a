"""ict_track_batch_from on the B200: what a start pose costs, and what it buys (DESIGN.md §6).

  cost   ict_track_batch and ict_track_batch_from with p_start = p_ref and with p_start != p_ref, called alternately in
         one process, median host time of the synchronous call over --reps rounds after --warmup rounds, on three
         workloads (4096 four-point 32x32 tracks at 1080p, 256 hundred-point 8x8 tracks at 640x480, dense 1080p) in
         sum orders 1 and 0;
  basin  fraction of 64 tracks (8 textured planes x 8 motions of synth.make_pair) that land within --tol of p_gt
         against the motion scale, for three strategies: from p_ref = 0, from p_gt perturbed by --frac of the motion
         (a prediction), and multi-start (each track's points replicated K = 8 times, one start each: 0 and seven
         draws of the motion prior at that scale, the result with the least evaluate() residual per visible point).

    python profiles/tools/from_time.py [--out results.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import invcompcamtrack_b200 as ict  # noqa: E402
from helpers import make_case  # noqa: E402
import test_gpu_track_from as F  # noqa: E402


def card():
    import torch
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch=torch.cuda.get_device_name(0), nvidia_smi=r.stdout.strip().splitlines()[:1])


def workload(name):
    if name == "4096x4pt-psz32-1080p":
        return make_case(seed=17, w=1920, h=1080, psz=32, npts=4, ntracks=4096)
    if name == "256x100pt-psz8-640x480":
        return make_case(seed=11, w=640, h=480, psz=8, npts=100, ntracks=256)
    return make_case(seed=21, w=1920, h=1080, psz=1, lv_f=3, dense_border=16)


def cost(name, order, warmup, reps):
    c = workload(name)
    tr, fr = F.open_case(ict, c, order)
    T = c["T"]
    p_ref = np.zeros((T, 6))
    s = 640.0 / c["w"]
    p_other = p_ref + np.array([0.01, -0.01, 0.005, 0.001, -0.001, 0.0005]) * s
    calls = {"track_batch": lambda: tr.track_batch(fr, 0, 1, p_ref),
             "from p_start=p_ref": lambda: tr.track_batch(fr, 0, 1, p_ref, p_start=p_ref),
             "from p_start!=p_ref": lambda: tr.track_batch(fr, 0, 1, p_ref, p_start=p_other)}
    times = {k: [] for k in calls}
    try:
        for rep in range(warmup + reps):
            for k, f in calls.items():
                t0 = time.perf_counter()
                f()                                   # returns after the device synchronise
                if rep >= warmup:
                    times[k].append(time.perf_counter() - t0)
    finally:
        tr.close()
        fr.close()
    res = {k: dict(median_ms=1e3 * float(np.median(v)), min_ms=1e3 * float(np.min(v)), max_ms=1e3 * float(np.max(v)))
           for k, v in times.items()}
    print(name, "order", order, json.dumps(res), flush=True)
    return res


def basin(scales, orders, frac, tol, K=8):
    scenes = F.gt_scenes()
    out = []
    for order in orders:
        for S in scales:
            frames, rf, nf, pts, p_gt = F.gt_pairs(scenes, S)
            T = F.GT_TRACKS
            zero = np.zeros((T, 6))
            tr, fr = F.gt_tracker(ict, scenes, frames, order, pts)
            try:
                e_ref = F.gt_error(tr.track_batch(fr, rf, nf, zero)["p_out"], p_gt)
                e_pred = F.gt_error(tr.track_batch(fr, rf, nf, zero, p_start=F.gt_prediction(p_gt, frac))["p_out"],
                                    p_gt)
            finally:
                tr.close()
                fr.close()
            # multi-start: K copies of each track, start k = 0 (k = 0) or a draw of the motion prior at scale S
            sc = scenes[0][0]
            starts = np.zeros((T, K, 6))
            for t in range(T):
                for k in range(1, K):
                    starts[t, k] = sc.random_motion(50000 + 97 * t + k, S)
            tr, fr = F.gt_tracker(ict, scenes, frames, order, pts, copies=K)
            try:
                rfk, nfk = np.repeat(rf, K), np.repeat(nf, K)
                zk = np.zeros((T * K, 6))
                out_k = tr.track_batch(fr, rfk, nfk, zk, p_start=starts.reshape(-1, 6))["p_out"]
                ev = tr.evaluate(fr, rfk, nfk, zk, p_cur=out_k)
            finally:
                tr.close()
                fr.close()
            score = np.where(ev["nvis"] > 0, ev["ssr"] / np.maximum(ev["nvis"], 1), np.inf).reshape(T, K)
            pick = out_k.reshape(T, K, 6)[np.arange(T), np.argmin(score, 1)]
            e_multi = F.gt_error(pick, p_gt)
            row = dict(order=order, scale=S, flow_px_max=float(np.abs(p_gt[:, :3]).max() * F.GT_W / 5.0),
                       from_ref=float((e_ref <= tol).mean()), from_prediction=float((e_pred <= tol).mean()),
                       multi_start=float((e_multi <= tol).mean()),
                       err_ref_median=float(np.median(e_ref)), err_pred_max=float(e_pred.max()))
            print(json.dumps(row), flush=True)
            row.update(err_ref=e_ref.tolist(), err_pred=e_pred.tolist(), err_multi=e_multi.tolist())
            out.append(row)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the results (JSON) there")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--frac", type=float, default=F.GT_FRAC)
    ap.add_argument("--tol", type=float, default=F.GT_TOL)
    ap.add_argument("--scales", default="1,2,3,4,6,8,10,12")
    ap.add_argument("--no-cost", action="store_true")
    ap.add_argument("--no-basin", action="store_true")
    a = ap.parse_args()
    ict.lib().ict_set_device(0)
    res = dict(card=card())
    print(json.dumps(res), flush=True)
    if not a.no_cost:
        res["cost"] = {"%s order %d" % (w, o): cost(w, o, a.warmup, a.reps)
                       for w in ("4096x4pt-psz32-1080p", "256x100pt-psz8-640x480", "dense-1080p") for o in (1, 0)}
    if not a.no_basin:
        res["basin"] = basin([float(x) for x in a.scales.split(",")], (1, 0), a.frac, a.tol)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
