#!/usr/bin/env python
"""bench.py — throughput of the inverse-compositional GN tracking path on B200 (one process per GPU).

Workload (BASELINE.json configs[4] per-GPU share == configs[2] geometry): S independent synthetic 1080p frame
pairs per GPU ("sequences" advancing one frame), T = 4096 independent tracks each, every track 4 points with
32x32 patches, 4-level pyramid, maxiter 10, normdp_ratio 0.01.  configs[1] (one 100-point template over 100
frames) cannot occupy a GPU and is a parity-test case (tests/test_gpu_parity.py::test_sequence_chain).

One step = for every local sequence: build the I/dx/dy pyramids of both frames on the device
(util_constructpyramide), then Set3Dpoints -> SetPose -> TrackPose for all S*T tracks (all levels, all GN
iterations, convergence test on device).
  value  : pixel-residuals/s with the uint8 frames, points and poses already resident in HBM, in the library's
           DEFAULT summation order = the reference's (bit-identical to the oracle; checked on the sampled tracks in
           every default run); `fast_mode` reports the opt-in tree-order kernels beside it
  e2e    : the same through the host-buffer C ABI (pinned host memory -> H2D -> kernels -> D2H) every step
  roofline: the tracking kernel, algorithmic 32 B per pixel-residual (SURVEY.md §8(d)) over its CUDA-event time
Weak scaling (default): per-GPU work is fixed.  --strong: the 256 sequences of BASELINE configs[4] are split over the
ranks.  Ranks share nothing on the hot path; poses are all-gathered (NCCL) once after the timed region (gather_ms).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the tree may be read-only: no byte-code caches written into it

BYTES_PER_PIXRES = 32.0   # 4 B pat_ref + 6*4 B steepest-descent values + 4 B new-frame texel (SURVEY.md §8(d))


def env_int(k, d):
    return int(os.environ.get(k, d))


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.idx, self.rows, self.stop_ev = gpu_index, [], threading.Event()

    def run(self):
        while not self.stop_ev.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([x.strip() for x in out.strip().split(",")])
            except Exception:
                pass
            self.stop_ev.wait(0.2)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[k] for r in self.rows if len(r) >= 7 for k in range(4) if r[3 + k].lower() == "active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def make_workload(rank, S, T, P, psz, w, h, lv_f, ntex):
    """S frame pairs (uint8) + S*T tracks of P plane points each; deterministic in (rank, s)."""
    from invcompcamtrack_b200 import synth
    scenes = {}
    frames = np.empty((2 * S, h, w), np.uint8)
    pts = np.empty(3 * S * T * P, np.float64)
    p_gt = np.zeros((S, 6))
    fc = cc = wh = None
    for s in range(S):
        gs = rank * S + s
        tex_id = gs % ntex
        if tex_id not in scenes:
            scenes[tex_id] = synth.Scene(tex_id, w, h)
        sc = scenes[tex_id]
        fc, cc, wh = sc.fc, sc.cc, sc.wh
        p_gt[s] = sc.random_motion(gs)
        frames[2 * s] = sc.render(np.zeros(6))
        frames[2 * s + 1] = sc.render(p_gt[s])
        # T tracks x P points: one draw of T*P points, regrouped per track as X block, Y block, Z block
        q = sc.points(gs, T * P, psz, lv_f).reshape(3, T, P)
        pts[3 * s * T * P:3 * (s + 1) * T * P] = np.ascontiguousarray(q.transpose(1, 0, 2)).reshape(-1)
    pt_off = np.arange(S * T + 1, dtype=np.int64) * P
    ref = np.repeat(np.arange(S, dtype=np.int32) * 2, T)
    new = ref + 1
    return dict(frames=frames, pts=pts, pt_off=pt_off, ref=ref, new=new, p_gt=p_gt, fc=fc, cc=cc, wh=wh)


def cpu_sample(wl, op_kw, S, T, P, psz, w, h, lv_f, seqs, threads, use_ref, spread=False):
    """Times the CPU implementation (oracle port or oracle/_ref) on `seqs` sequences of the same workload."""
    from oracle import oracle as O
    orc = O.OracleLib()
    op = O.make_optparam(**op_kw)
    seqs = min(seqs, S)
    t0 = time.perf_counter()
    pyr = [orc.pyramid_build(wl["frames"][f].astype(np.float32), lv_f, psz) for f in range(2 * seqs)]
    t_pyr = time.perf_counter() - t0
    n = seqs * T
    args = (op, wl["fc"], wl["cc"], wl["wh"], [q[0] for q in pyr], [q[1] for q in pyr], [q[2] for q in pyr],
            wl["pt_off"][:n + 1], wl["pts"][:3 * n * P].copy(), wl["ref"][:n], wl["new"][:n], np.zeros((n, 6)))
    # pixel-residual count always from the instrumented port (the reference classes do not expose it)
    counted = orc.track_batch(*args, nthreads=threads)
    npix = int(counted["npixres"].sum())
    if use_ref and O.RefLib.available():
        ref = O.RefLib()
        t0 = time.perf_counter()
        ref.track_batch(*args, nthreads=threads)
        dt = time.perf_counter() - t0
        kind = "reference"
    else:
        t0 = time.perf_counter()
        orc.track_batch(*args, nthreads=threads)
        dt = time.perf_counter() - t0
        kind = "port"
    alt = None
    if spread:
        # the same sample with the reference's sums in the other packet order its unpinned Eigen could have used
        # (AVX instead of SSE packets): how far the REFERENCE moves from itself when only that order changes
        orc.set_sum_mode(1)
        alt = orc.track_batch(*args, nthreads=threads)
        orc.set_sum_mode(0)
    return dict(value=npix / dt, tracks_per_s=n / dt, seconds=dt, kind=kind, npix=npix, tracks=n,
                pyramid_ms_per_frame=1e3 * t_pyr / (2 * seqs), p_out=counted["p_out"], iters=counted["iters"],
                alt=alt)


def _best_of(fn, reps):
    import torch
    best, out = None, None
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        dt = time.perf_counter() - t0
        best = dt if best is None or dt < best else best
    return best, out


def other_configs(ict, dev, cores):
    """The other BASELINE configs through the same library, each with its CPU baseline (oracle port, 1 thread and all
    cores), its parity against the oracle and the bound of its kernel: configs[0] single pair, configs[1] one
    100-point template chain over 100 frames, configs[3] dense full-frame alignment at 1080p."""
    import torch
    from invcompcamtrack_b200 import synth
    from oracle import oracle as O
    orc = O.OracleLib()
    peak, peak_src = read_peaks()
    out = {}

    def cpu_tracks(op_o, sc, pyr, pt_off, pts, ref, new, p_in, threads):
        t0 = time.perf_counter()
        r = orc.track_batch(op_o, sc.fc, sc.cc, sc.wh, [q[0] for q in pyr], [q[1] for q in pyr], [q[2] for q in pyr],
                            pt_off, pts.copy(), ref, new, p_in, nthreads=threads)
        return time.perf_counter() - t0, r

    # ---- configs[0]: run_track, one 100-point 8x8 template on a 640x480 pair (the reference's own timing size) ------
    sc, A, B, p_gt = synth.make_pair(7, 640, 480)
    pts = sc.points(911, 100, 8, 3)
    kw = dict(lv_f=3, lv_l=0, psz=8, maxiter=10, normdp_ratio=0.01, donorm=0, dopatchnorm=0, maxpttrack=100)
    op, op_o = ict.make_optparam(**kw), O.make_optparam(**kw)
    fr = ict.Frames(2, 640, 480, 3, 8)
    fr.upload(0, np.stack([A, B]))
    tr = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
    tr.set_points(np.array([0, 100], np.int64), pts.copy())
    t_ref, r = _best_of(lambda: tr.track_batch(fr, 0, 1, np.zeros((1, 6))), 5)
    tr.set_sum_order(0)
    t_fast, r0 = _best_of(lambda: tr.track_batch(fr, 0, 1, np.zeros((1, 6))), 5)
    pyr = [orc.pyramid_build(x.astype(np.float32), 3, 8) for x in (A, B)]
    t_cpu, ro = cpu_tracks(op_o, sc, pyr, np.array([0, 100], np.int64), pts, [0], [1], np.zeros((1, 6)), 1)
    t_cpu = min(t_cpu, cpu_tracks(op_o, sc, pyr, np.array([0, 100], np.int64), pts, [0], [1], np.zeros((1, 6)), 1)[0])
    npix = int(r["npixres"].sum())
    out["single_pair"] = {
        "workload": "BASELINE configs[0]: run_track, one 100-point 8x8 template, 640x480 pair, 4 levels (a latency case: "
                    "one track cannot occupy a GPU)",
        "ms_per_trackpose": 1e3 * t_ref, "value": npix / t_ref, "unit": "pixel-residuals/s",
        "fast_mode": {"ms_per_trackpose": 1e3 * t_fast, "value": int(r0["npixres"].sum()) / t_fast},
        "cpu_baseline": {"kind": "port", "cores": 1, "ms_per_trackpose": 1e3 * t_cpu, "value": int(ro["npixres"].sum()) / t_cpu,
                         "unit": "pixel-residuals/s", "sample": "the same track, oracle port, 1 thread (one track has no "
                         "parallelism on the CPU: the all-cores figure is the same)"},
        "parity": {"bit_identical_pose_and_iteration_counts": bool(np.array_equal(r["p_out"], ro["p_out"]) and
                                                                   np.array_equal(r["iters"], ro["iters"])),
                   "err_vs_ground_truth": float(np.abs(r["p_out"][0] - p_gt).max())},
        "roofline": {"bound": "latency", "note": "one CTA on one SM: host call + one launch + the sequential chains of "
                     "%d GN iterations; not a throughput case" % int(r["iters"].sum())}}
    tr.close(); fr.close()

    # ---- configs[1]: run_track_nposes-style chain, 100 frames, 640x480, psz 8, 100 points; 256 pose samples ----------
    NF, S = 100, 256
    sc, frames, poses = synth.make_sequence(5, NF, 640, 480)
    fr = ict.Frames(NF, 640, 480, 3, 8)
    fr.upload(0, np.stack(frames))
    tr = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
    cpts = np.concatenate([sc.points(100 + s_, 100, 8, 3) for s_ in range(S)])
    tr.set_points(np.arange(S + 1, dtype=np.int64) * 100, cpts.copy())
    t_ref, r = _best_of(lambda: tr.track_sequence(fr, 0, NF - 1, 1, np.zeros((S, 6))), 2)
    tr.set_sum_order(0)
    t_fast, r0 = _best_of(lambda: tr.track_sequence(fr, 0, NF - 1, 1, np.zeros((S, 6))), 2)
    # CPU: bounded sample — CS chains over CF frame steps, chained like run_track_nposes.cpp:232-239
    CS, CF = 16, 12
    pyr = [orc.pyramid_build(f.astype(np.float32), 3, 8) for f in frames[:CF + 1]]
    off = np.arange(CS + 1, dtype=np.int64) * 100
    cpu = {}
    for threads in (1, cores):
        p = np.zeros((CS, 6)); tot = 0.0; npx = 0; chain = [p.copy()]
        for k in range(CF):
            dt, ro = cpu_tracks(op_o, sc, pyr, off, cpts[:300 * CS], np.full(CS, k, np.int32), np.full(CS, k + 1, np.int32), p, threads)
            tot += dt; npx += int(ro["npixres"].sum()); p = ro["p_out"]; chain.append(p.copy())
        cpu[threads] = (npx / tot, CS * CF / tot)
    same = all(np.array_equal(r["poses"][k, :CS], chain[k]) for k in range(CF + 1))
    out["chain_100_frames"] = {
        "workload": "BASELINE configs[1]: %d pose samples x one 100-point template chained over %d frames of 640x480, psz 8, "
                    "4 levels" % (S, NF),
        "ms_per_chain_batch": 1e3 * t_ref, "tracks_per_s": S * (NF - 1) / t_ref, "value": int(r["npixres"].sum()) / t_ref,
        "unit": "pixel-residuals/s",
        "fast_mode": {"ms_per_chain_batch": 1e3 * t_fast, "tracks_per_s": S * (NF - 1) / t_fast,
                      "value": int(r0["npixres"].sum()) / t_fast},
        "cpu_baseline": {"kind": "port", "unit": "pixel-residuals/s", "value_1_thread": cpu[1][0], "tracks_per_s_1_thread": cpu[1][1],
                         "cores": cores, "value": cpu[cores][0], "tracks_per_s": cpu[cores][1],
                         "sample": "%d of the %d chains over the first %d of the %d frame steps" % (CS, S, CF, NF - 1)},
        "parity": {"bit_identical_poses_on_cpu_sample": bool(same),
                   "drift_vs_ground_truth": float(np.abs(r["poses"][-1, 0] - poses[-1]).max())},
        "roofline": {"bound": "hbm", "achieved": 32.0 * int(r["npixres"].sum()) / t_ref / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": 32.0 * int(r["npixres"].sum()) / t_ref / 1e9 / peak,
                     "note": "algorithmic 32 B per pixel-residual over the host call; the template is resident on chip, the "
                             "kernel (k_track_x8) is bound by its sequential fp32 chains, not by HBM"}}
    tr.close(); fr.close()

    # ---- configs[3]: dense, one point per pixel, psz 1, tilted plane (per-pixel depth) ----------------------------
    w, h = 1920, 1080
    sc, A, B, p_gt = synth.make_pair(41, w, h, tilt=(0.05, -0.03))
    pts = sc.dense_points(16)
    n = pts.size // 3
    kw = dict(lv_f=3, lv_l=0, psz=1, maxiter=10, normdp_ratio=0.01, donorm=0, dopatchnorm=0, maxpttrack=n)
    op, op_o = ict.make_optparam(**kw), O.make_optparam(**kw)
    fr = ict.Frames(2, w, h, 3, 1)
    fr.upload(0, np.stack([A, B]))
    tr = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
    tr.set_points(np.array([0, n], np.int64), pts.copy())
    t_ref, r = _best_of(lambda: tr.track_batch(fr, 0, 1, np.zeros((1, 6))), 3)      # reference order (library default)
    tr.set_sum_order(0)
    t_fast, r0 = _best_of(lambda: tr.track_batch(fr, 0, 1, np.zeros((1, 6))), 4)    # fused streaming kernels
    npix, npix0 = int(r["npixres"].sum()), int(r0["npixres"].sum())
    pyr = [orc.pyramid_build(x.astype(np.float32), 3, 1) for x in (A, B)]
    t_cpu, ro = cpu_tracks(op_o, sc, pyr, np.array([0, n], np.int64), pts, [0], [1], np.zeros((1, 6)), 1)
    out["dense_1080p"] = {
        "workload": "BASELINE configs[3]: %d points (one per pixel), psz 1, 4 levels, %d GN iterations" % (n, int(r["iters"].sum())),
        "ms_per_trackpose": 1e3 * t_ref, "value": npix / t_ref, "unit": "pixel-residuals/s",
        "fast_mode": {"ms_per_trackpose": 1e3 * t_fast, "value": npix0 / t_fast, "algorithmic_GBps": 44.0 * npix0 / t_fast / 1e9,
                      "frac_of_hbm_peak": 44.0 * npix0 / t_fast / 1e9 / peak,
                      "note": "fused streaming kernels (k_dense_level / k_dense_iter_tma), tree sums; whole host call"},
        "cpu_baseline": {"kind": "port", "cores": 1, "ms_per_trackpose": 1e3 * t_cpu, "value": int(ro["npixres"].sum()) / t_cpu,
                         "unit": "pixel-residuals/s", "sample": "the same TrackPose, oracle port, 1 thread (one track: the "
                         "reference has no parallelism inside a track)"},
        "parity": {"bit_identical_pose_and_iteration_counts": bool(np.array_equal(r["p_out"], ro["p_out"]) and
                                                                   np.array_equal(r["iters"], ro["iters"])),
                   "fast_mode_max_abs_pose_diff": float(np.abs(r0["p_out"] - ro["p_out"]).max()),
                   "fast_mode_identical_iteration_counts": bool(np.array_equal(r0["iters"], ro["iters"]))},
        "roofline": {"bound": "hbm", "achieved": 44.0 * npix / t_ref / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": 44.0 * npix / t_ref / 1e9 / peak, "algorithmic_bytes_per_pixel_residual": 44,
                     "note": "whole TrackPose host call in the reference order (44 B per pixel-residual, SURVEY.md 8d)"}}
    tr.close()
    # the streaming iteration kernel alone: slope between runs of 2 and 10 iterations per level (the stop rule off)
    tt = {}
    for mi in (2, 10):
        op2 = ict.make_optparam(lv_f=3, lv_l=0, psz=1, maxiter=mi, normdp_ratio=1e-30, donorm=0, dopatchnorm=0, maxpttrack=n)
        tr = ict.Tracker(op2, sc.fc, sc.cc, sc.wh)
        tr.set_sum_order(0)
        tr.set_points(np.array([0, n], np.int64), pts.copy())
        tt[mi], _ = _best_of(lambda: tr.track_batch(fr, 0, 1, np.zeros((1, 6))), 5)
        tr.close()
    per_it = (tt[10] - tt[2]) / 32.0
    out["dense_1080p"]["fast_mode"]["iteration_kernel"] = {
        "name": "k_dense_iter_tma<3>", "us_per_launch": 1e6 * per_it, "bytes_per_point": 44,
        "achieved_GBps": 44.0 * n / per_it / 1e9, "peak_GBps": peak, "frac": 44.0 * n / per_it / 1e9 / peak,
        "fixed_us_per_trackpose": 1e6 * (tt[2] - 8 * per_it),
        "method": "(t[10 iterations/level] - t[2 iterations/level]) / 32 launches, stop rule off; includes launch and "
                  "the last CTA's solve; 44 B per point = 40 B streamed (X, Y, Z, ref, sd1..6) + one 4 B texel "
                  "(SURVEY.md 8d)"}
    fr.close()
    return out


KERNEL_NAME = "k_track_r<4,2>"   # the reference-order kernel for psz 32, up to 4 points per track (ict_kernel_r.cu)
DUMP_BYTES = 60 * 10 ** 6           # --dump-outputs stays below 64 MB, .npy headers included


def dump_outputs(out_dir, arrays, suffix=""):
    """Writes per-track arrays (first axis = track) as <out_dir>/<name><suffix>.npy in float64, at most DUMP_BYTES in
    all: above that, the rows of a fixed seeded sample of tracks, whose indices go to track_index<suffix>.npy."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(a, np.float64) for k, a in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = 8 * sum(a[0].size for a in arrays.values())
    if n * row_bytes > DUMP_BYTES:
        idx = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // (row_bytes + 8), replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        arrays["track_index"] = idx.astype(np.float64)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + suffix + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--seqs", type=int, default=env_int("ICT_BENCH_SEQS", 32), help="sequences (frame pairs) per GPU")
    ap.add_argument("--tracks", type=int, default=4096, help="tracks per sequence")
    ap.add_argument("--points", type=int, default=4, help="points per track")
    ap.add_argument("--psz", type=int, default=32)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--cpu-seqs", type=int, default=env_int("ICT_BENCH_CPU_SEQS", 8), help="sequences in the CPU sample")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-chunks", type=int, default=env_int("ICT_BENCH_E2E_CHUNKS", 4),
                    help="chunks of sequences the host-buffer path pipelines over two streams")
    ap.add_argument("--maxiter", type=int, default=10)
    ap.add_argument("--ratio", type=float, default=0.01, help="normdp_ratio")
    ap.add_argument("--textures", type=int, default=4, help="distinct textures shared by the sequences (setup time)")
    ap.add_argument("--strong", action="store_true",
                    help="strong scaling: the 256 sequences of BASELINE configs[4] in total, split over the ranks")
    ap.add_argument("--no-fast", action="store_true", help="skip the fast_mode (tree-order kernels) leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the poses, iteration counts and pixel-residual counts of the last timed step as "
                         "DIR/p_out.npy, iters.npy, npixres.npy (float64, one row per track)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")

    rank, world = env_int("RANK", 0), env_int("WORLD_SIZE", 1)
    local_rank = env_int("LOCAL_RANK", 0)
    if a.strong:
        a.seqs = max(1, 256 // world)
    S, T, P, psz, w, h, lv_f = a.seqs, a.tracks, a.points, a.psz, a.width, a.height, 3
    op_kw = dict(lv_f=lv_f, lv_l=0, psz=psz, maxiter=a.maxiter, normdp_ratio=a.ratio, donorm=0, dopatchnorm=0, maxpttrack=P)
    config = {"workload": "S=%d synthetic %dx%d frame pairs x %d tracks x %d points x %dx%d patches per GPU, "
                          "4-level pyramid, maxiter %d, normdp_ratio %g (BASELINE configs[4] per-GPU share%s); "
                          "reference summation order (library default, bit-identical to the oracle)"
                          % (S, w, h, T, P, psz, psz, a.maxiter, a.ratio, ", --strong: 256 sequences in total" if a.strong else ""),
              "seqs_per_gpu": S, "tracks_per_seq": T, "points_per_track": P, "psz": psz, "frame": [w, h],
              "levels": lv_f + 1, "l2_policy": "inputs larger than L2: %.0f MB of pyramids + %.0f MB of uint8 frames per step"
              % (S * 2 * 3 * 12.52, S * 2 * w * h / 1e6)}
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)

    # ------------------------------------------------------------------------------------------------
    if a.impl == "reference":
        # the reference's own CPU implementation on the host cores: rank 0 only, bounded sample per step
        if rank != 0:
            return 0
        from oracle import oracle as O
        use_ref = O.RefLib.available()
        seqs = max(1, min(a.cpu_seqs, S))
        wl = make_workload(0, seqs, T, P, psz, w, h, lv_f, a.textures)
        times, res = [], None
        for k in range(a.warmup + a.steps):
            res = cpu_sample(wl, op_kw, seqs, T, P, psz, w, h, lv_f, seqs, cores, use_ref)
            if k >= a.warmup:
                times.append(res["seconds"])
        dt = float(np.mean(times))
        val = res["npix"] / dt
        sample = ("%d sequences x %d tracks per step (of %d per GPU); %s; span Set3Dpoints->SetPose->TrackPose, "
                  "pyramids built beforehand (%.1f ms/frame, 1 thread)"
                  % (seqs, T, S, "reference sources (utilities/camera/pose/odometer.cpp) compiled against the stand-in "
                     "Eigen/OpenCV headers of oracle/shim" if res["kind"] == "reference" else "oracle port (plain C)",
                     res["pyramid_ms_per_frame"]))
        line = {"impl": "reference", "metric": "GN pixel-residuals/s", "value": val, "unit": "pixel-residuals/s",
                "tracks_per_s": res["tracks"] / dt, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": 1e3 * dt, "higher_is_better": True, "scaling": "strong" if a.strong else "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": val, "unit": "pixel-residuals/s", "cores": cores, "kind": res["kind"],
                                 "sample": sample},
                "e2e": {"value": val, "unit": "pixel-residuals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------------------------------------
    import torch
    import torch.distributed as dist
    import invcompcamtrack_b200 as ict

    if not torch.cuda.is_available() or ict.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device — the tracking path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    ict.lib().ict_set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    wl = make_workload(rank, S, T, P, psz, w, h, lv_f, a.textures)
    NT = S * T
    L = lv_f + 1
    op = ict.make_optparam(**op_kw)
    frames = ict.Frames(2 * S, w, h, lv_f, psz)
    tracker = ict.Tracker(op, wl["fc"], wl["cc"], wl["wh"])

    # device-resident inputs
    d_frames = torch.from_numpy(wl["frames"]).to(dev)
    d_pts = torch.from_numpy(wl["pts"]).to(dev)
    d_off = torch.from_numpy(wl["pt_off"]).to(dev)
    d_ref = torch.from_numpy(wl["ref"]).to(dev)
    d_new = torch.from_numpy(wl["new"]).to(dev)
    d_pin = torch.zeros(NT, 6, dtype=torch.float64, device=dev)
    d_pout = torch.zeros(NT, 6, dtype=torch.float64, device=dev)
    d_iters = torch.zeros(NT, L, dtype=torch.int32, device=dev)
    d_npix = torch.zeros(NT, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    ev_k0 = [torch.cuda.Event(enable_timing=True) for _ in range(a.steps)]
    ev_k1 = [torch.cuda.Event(enable_timing=True) for _ in range(a.steps)]

    def step_dev(k=None):
        frames.build_dev(0, 2 * S, d_frames.data_ptr(), u8=True, stream=stream)
        tracker.set_points_dev(NT, d_off.data_ptr(), d_pts.data_ptr(), NT * P, P, stream=stream)
        if k is not None:
            ev_k0[k].record()
        tracker.track_batch_dev(frames, d_ref.data_ptr(), d_new.data_ptr(), d_pin.data_ptr(), d_pout.data_ptr(),
                                iters_ptr=d_iters.data_ptr(), npix_ptr=d_npix.data_ptr(), stream=stream)
        if k is not None:
            ev_k1[k].record()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(a.warmup):
        step_dev()
    barrier()
    ict.launch_count(reset=True)
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(a.steps):
        step_dev(k)
    e1.record()
    barrier()
    launches = ict.launch_count()
    ms_total = e0.elapsed_time(e1)
    ms_kernel = float(np.mean([ev_k0[k].elapsed_time(ev_k1[k]) for k in range(a.steps)]))
    npix_step = int(d_npix.sum().item())
    iters_mean = float(d_iters.sum(dim=1).double().mean().item())
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"p_out": d_pout.cpu().numpy(), "iters": d_iters.cpu().numpy(),
                                      "npixres": d_npix.cpu().numpy()}, "_rank%d" % rank if world > 1 else "")

    # ---- fast mode (opt-in tree-order kernels), device-resident, same workload: reported beside the headline -----
    fast = None
    if not a.no_fast:
        tr_f = ict.Tracker(op, wl["fc"], wl["cc"], wl["wh"])
        tr_f.set_sum_order(0)
        f_pout = torch.zeros(NT, 6, dtype=torch.float64, device=dev)
        f_iters = torch.zeros(NT, L, dtype=torch.int32, device=dev)
        f_npix = torch.zeros(NT, dtype=torch.int64, device=dev)

        def step_fast():
            frames.build_dev(0, 2 * S, d_frames.data_ptr(), u8=True, stream=stream)
            tr_f.set_points_dev(NT, d_off.data_ptr(), d_pts.data_ptr(), NT * P, P, stream=stream)
            tr_f.track_batch_dev(frames, d_ref.data_ptr(), d_new.data_ptr(), d_pin.data_ptr(), f_pout.data_ptr(),
                                 iters_ptr=f_iters.data_ptr(), npix_ptr=f_npix.data_ptr(), stream=stream)

        for _ in range(2):
            step_fast()
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(a.steps):
            step_fast()
        g1.record()
        barrier()
        fast = dict(ms=g0.elapsed_time(g1) / a.steps, npix=int(f_npix.sum().item()), pout=f_pout, iters=f_iters)
        tr_f.close()

    # ---- e2e: host buffers through the C ABI, H2D/D2H inside the timed region ----------------------------
    e2e = None
    if not a.no_e2e:
        h_frames = torch.from_numpy(wl["frames"]).pin_memory()
        h_pts = torch.from_numpy(wl["pts"]).pin_memory()
        h_pin = torch.zeros(NT, 6, dtype=torch.float64).pin_memory()
        h_pout = torch.zeros(NT, 6, dtype=torch.float64).pin_memory()
        h_iters = torch.zeros(NT, L, dtype=torch.int32).pin_memory()
        h_npix = torch.zeros(NT, dtype=torch.int64).pin_memory()
        import ctypes as C
        lib = ict.lib()
        v = C.c_void_p

        # The batch goes through the C ABI in chunks of sequences on ONE stream, one tracker per chunk: the *_stream
        # entry points run their host->device copies on internal copy lanes, so the copy of chunk c+1 overlaps the
        # tracking of chunk c while all kernels stay in call order on this stream (two caller streams made the
        # pyramid kernel of the next chunk run inside the tracking kernel at a fraction of its occupancy).
        nchunk = max(1, min(a.e2e_chunks, S))
        bounds = [(c * S) // nchunk for c in range(nchunk + 1)]
        streams = [torch.cuda.Stream()]
        chunk_trackers = [ict.Tracker(op, wl["fc"], wl["cc"], wl["wh"]) for _ in range(nchunk)]
        # every host buffer the ABI reads asynchronously is pinned (a pageable source makes cudaMemcpyAsync wait for
        # the stream and serialises the pipeline)
        h_ref = torch.from_numpy(wl["ref"]).pin_memory()
        h_new = torch.from_numpy(wl["new"]).pin_memory()
        chunk_off = []
        for c in range(nchunk):
            t0_, t1_ = bounds[c] * T, bounds[c + 1] * T
            chunk_off.append(torch.from_numpy(np.ascontiguousarray(wl["pt_off"][t0_:t1_ + 1] - wl["pt_off"][t0_])).pin_memory())

        def step_host():
            for c in range(nchunk):
                st = v(streams[0].cuda_stream)
                s0, s1 = bounds[c], bounds[c + 1]
                t0_, t1_ = s0 * T, s1 * T
                rc = lib.ict_frames_upload_u8_stream(frames.h_, 2 * s0, 2 * (s1 - s0),
                                                     v(h_frames.data_ptr() + 2 * s0 * w * h), st)
                rc |= lib.ict_tracker_set_points_stream(chunk_trackers[c].h_, t1_ - t0_, v(chunk_off[c].data_ptr()),
                                                        v(h_pts.data_ptr() + 8 * 3 * int(wl["pt_off"][t0_])), st)
                rc |= lib.ict_track_batch_stream(chunk_trackers[c].h_, frames.h_, v(h_ref.data_ptr() + 4 * t0_),
                                                 v(h_new.data_ptr() + 4 * t0_), v(h_pin.data_ptr() + 48 * t0_),
                                                 v(h_pout.data_ptr() + 48 * t0_), v(h_iters.data_ptr() + 4 * L * t0_),
                                                 v(h_npix.data_ptr() + 8 * t0_), st)
                if rc:
                    raise ict.IctError(lib.ict_last_error().decode())

        def fork():
            ev = torch.cuda.Event()
            ev.record()
            for st_ in streams:
                st_.wait_event(ev)

        def join():
            for st_ in streams:
                ev = torch.cuda.Event()
                ev.record(st_)
                torch.cuda.current_stream().wait_event(ev)

        fork()
        for _ in range(min(a.warmup, 2)):
            step_host()
        join()
        barrier()
        t0 = time.perf_counter()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        fork()
        for _ in range(a.steps):
            step_host()
        join()
        f1.record()
        barrier()
        wall = time.perf_counter() - t0
        ms_e2e = max(f0.elapsed_time(f1), 0.0)
        if not torch.equal(h_pout.to(dev), d_pout):
            raise SystemExit("bench.py: host-buffer path and device-resident path disagree")
        h2d = h_frames.numel() + 8 * h_pts.numel() + 8 * wl["pt_off"].size + 4 * 2 * NT + 48 * NT
        d2h = 48 * NT + 4 * L * NT + 8 * NT
        e2e = dict(ms=ms_e2e, wall_ms=1e3 * wall, h2d=int(h2d), d2h=int(d2h), npix=int(h_npix.sum().item()))
    clocks = None
    sampler.stop_ev.set()
    sampler.join(timeout=3)
    clocks = sampler.summary()

    # ---- max over ranks, whole-job aggregate ------------------------------------------------------------
    stats = torch.tensor([ms_total, ms_kernel, e2e["ms"] if e2e else 0.0, float(npix_step),
                          fast["ms"] if fast else 0.0, float(fast["npix"]) if fast else 0.0], dtype=torch.float64, device=dev)
    gather_ms = None
    if world > 1:
        mx = stats.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stats.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        # the one collective of the path: gather the per-track poses (6 f64) and iteration counts, once
        from invcompcamtrack_b200.shard import gather_results
        gather_results(d_pout, d_iters)           # warm-up (communicator set-up)
        barrier()
        q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        q0.record()
        all_poses, all_iters = gather_results(d_pout, d_iters)
        q1.record()
        torch.cuda.synchronize()
        assert all_poses.shape[0] == NT * world
        gms = torch.tensor([q0.elapsed_time(q1)], dtype=torch.float64, device=dev)
        dist.all_reduce(gms, op=dist.ReduceOp.MAX)
        gather_ms = gms.item()
        ms_total, ms_kernel, ms_e2e_all, ms_fast = mx[0].item(), mx[1].item(), mx[2].item(), mx[4].item()
        npix_job, npix_fast_job = sm[3].item(), sm[5].item()
    else:
        ms_e2e_all = e2e["ms"] if e2e else 0.0
        npix_job = float(npix_step)
        ms_fast, npix_fast_job = (fast["ms"], float(fast["npix"])) if fast else (0.0, 0.0)

    if rank == 0:
        peak, peak_src = read_peaks()
        value = npix_job * a.steps / (ms_total * 1e-3)
        tracks_s = NT * world * a.steps / (ms_total * 1e-3)
        achieved = npix_step * BYTES_PER_PIXRES / (ms_kernel * 1e-3) / 1e9
        # counters of the tracking kernel from this round's ncu capture (profiles/, committed): DRAM traffic per track,
        # issue slots, shared-memory pipe — what actually bounds the kernel; never measured under the bench's own clock
        counters, traffic = None, None
        cp = os.path.join(ROOT, "profiles", "r02_k_track_r_counters.json")
        if os.path.exists(cp):
            try:
                counters = json.load(open(cp))
                traffic = counters["dram_bytes_per_track"] * NT          # per launch, like `achieved`
            except Exception:
                counters, traffic = None, None
        line = {"metric": "GN pixel-residuals/s", "value": value, "unit": "pixel-residuals/s",
                "tracks_per_s": tracks_s, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": ms_total / a.steps, "higher_is_better": True, "scaling": "strong" if a.strong else "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "sum_order": "reference (Eigen 3.3 packet order; library default): bit-identical to the oracle",
                "pixel_residuals_per_step_per_gpu": npix_step, "gn_iterations_per_track": iters_mean,
                "roofline": {"bound": "hbm", "kernel": KERNEL_NAME if (psz == 32 and P <= 4) else "k_track (see DESIGN.md)",
                             "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "algorithmic_hbm_frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                             "algorithmic_bytes_per_pixel_residual": BYTES_PER_PIXRES,
                             "kernel_ms_per_launch": ms_kernel,
                             "kernel_share_of_step": ms_kernel / (ms_total / a.steps),
                             "limiter": "not HBM: the steepest-descent images are resident in shared memory; the kernel is "
                                        "bound by the reference order itself (8 sequential fp32 chains per sum, 4 cycles "
                                        "per addition) and by the rate at which one warp gets shared-memory loads issued "
                                        "(DESIGN.md §4, profiles/r02_k_track_r_ncu_summary.txt)",
                             "counters": counters,
                             "note": "achieved/frac = ALGORITHMIC bytes (32 B per pixel-residual, SURVEY.md 8d) over the kernel's "
                                     "CUDA-event time, as north_star defines the figure; `traffic` = measured DRAM bytes of "
                                     "the kernel (ncu, per track x tracks per launch) — far below the algorithmic bytes "
                                     "because the template never leaves the chip. The HBM-streaming kernel of the path is "
                                     "the dense iteration (other_configs.dense_1080p.fast_mode.iteration_kernel)"},
                "gpu_launches": int(launches), "clocks": clocks}
        if gather_ms is not None:
            line["gather_ms"] = gather_ms
            line["gather_note"] = ("one NCCL all-gather of 6 f64 + %d i32 per track over all ranks, after the timed region "
                                   "(the path's only collective)" % L)
        if fast:
            line["fast_mode"] = {"value": npix_fast_job / (ms_fast * 1e-3), "unit": "pixel-residuals/s",
                                 "ms_per_step": ms_fast, "tracks_per_s": NT * world / (ms_fast * 1e-3),
                                 "kernel": "k_track_v2 (ict_tracker_set_sum_order(tr, 0): tree sums, factorised J^T r)",
                                 "note": "opt-in; same step (pyramids + Set3Dpoints + tracking), inputs resident; NOT the "
                                         "headline because its iteration counts equal the oracle's on ~90 % of these "
                                         "4-point tracks only (parity_vs_gpu.fast_mode_kernel)"}
        if e2e:
            line["e2e"] = {"value": npix_job * a.steps / (ms_e2e_all * 1e-3), "unit": "pixel-residuals/s",
                           "h2d_bytes_per_step": e2e["h2d"], "d2h_bytes_per_step": e2e["d2h"],
                           "ms_per_step": ms_e2e_all / a.steps, "wall_ms_per_step": e2e["wall_ms"] / a.steps,
                           "tracks_per_s": NT * world * a.steps / (ms_e2e_all * 1e-3)}
        if world == 1 and not a.no_cpu:
            seqs = max(1, min(a.cpu_seqs, S))
            cb = cpu_sample(wl, op_kw, S, T, P, psz, w, h, lv_f, seqs, cores, use_ref=False, spread=True)
            cb1 = cpu_sample(wl, op_kw, S, T, P, psz, w, h, lv_f, 1, 1, use_ref=False)       # one thread: the reference as shipped
            # parity of the benchmark's own result against the oracle on the sampled tracks: the headline kernel runs
            # the reference's summation order, so poses and iteration counts must be EQUAL
            n = cb["tracks"]
            g = d_pout[:n].cpu().numpy()
            gi_ = d_iters[:n].cpu().numpy()
            exact = bool(np.array_equal(g, cb["p_out"]) and np.array_equal(gi_, cb["iters"]))
            same = float((gi_ == cb["iters"]).all(axis=1).mean())
            da = np.abs(cb["alt"]["p_out"] - cb["p_out"]).max(axis=1)
            same_alt = float((cb["alt"]["iters"] == cb["iters"]).mean())
            pv = {"note": "headline kernel = reference summation order: bit-identical to the oracle on every sampled track. "
                          "4-point tracks are ill-conditioned: the reference itself moves by reference_self_spread when only "
                          "the packet width of its own Eigen sums changes (oracle, SSE vs AVX packets) — the fast mode "
                          "differs from the oracle by as much",
                  "headline_kernel": {"bit_identical_poses_and_iteration_counts": exact, "tracks": int(n),
                                      "frac_tracks_identical_iteration_counts": same,
                                      "max_abs_pose_diff": float(np.abs(g - cb["p_out"]).max())},
                  "reference_self_spread": {"frac_identical_iteration_counts": same_alt,
                                            "median_abs_pose_diff": float(np.median(da)),
                                            "p99_abs_pose_diff": float(np.percentile(da, 99)),
                                            "max_abs_pose_diff": float(da.max())}}
            if fast:
                fg = fast["pout"][:n].cpu().numpy()
                dg = np.abs(fg - cb["p_out"]).max(axis=1)
                pv["fast_mode_kernel"] = {"frac_identical_iteration_counts": float((fast["iters"][:n].cpu().numpy() == cb["iters"]).mean()),
                                          "median_abs_pose_diff": float(np.median(dg)),
                                          "p99_abs_pose_diff": float(np.percentile(dg, 99)),
                                          "max_abs_pose_diff": float(dg.max())}
            line["cpu_baseline"] = {
                "value": cb["value"], "unit": "pixel-residuals/s", "cores": cores, "kind": cb["kind"],
                "tracks_per_s": cb["tracks_per_s"],
                "value_1_thread": cb1["value"], "tracks_per_s_1_thread": cb1["tracks_per_s"],
                "sample": "%d of the %d sequences (%d tracks), %.1f s, oracle port (plain C, -O3 -msse4 -mavx), OpenMP "
                          "over tracks on %d threads; 1-thread figure (the reference as shipped is single-threaded): 1 "
                          "sequence, %.1f s; span Set3Dpoints->SetPose->TrackPose; pyramids %.1f ms/frame on 1 thread extra"
                          % (seqs, S, cb["tracks"], cb["seconds"], cores, cb1["seconds"], cb["pyramid_ms_per_frame"]),
                "parity_vs_gpu": pv}
            try:
                line["other_configs"] = other_configs(ict, dev, cores)
            except Exception as e:          # secondary numbers must never cost the headline line
                line["other_configs"] = {"error": repr(e)}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
