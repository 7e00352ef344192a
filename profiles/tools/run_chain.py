"""BASELINE config 2: one 100-point template chain over a 100-frame 640x480 sequence (psz 8, 4 levels), S samples in
parallel (the `sid` loop of run_track_nposes.cpp:193 is the batch dimension); timing of ict_track_sequence."""
import os, sys, time
R = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))); sys.path.insert(0, R)
import numpy as np
import invcompcamtrack_b200 as ict
from invcompcamtrack_b200 import synth
from oracle import oracle as O
NF, S = int(os.environ.get("FRAMES", 100)), int(os.environ.get("SAMPLES", 1))
NP = int(os.environ.get("NPTS", 100))
sc, frames, poses = synth.make_sequence(5, NF, 640, 480)
op_c = O.make_optparam(lv_f=3, lv_l=0, psz=8, maxiter=10, normdp_ratio=0.01, donorm=int(os.environ.get('DONORM', 0)),
                        dopatchnorm=int(os.environ.get('PATCHNORM', 0)), maxpttrack=NP)
op = ict.OptParam.from_buffer_copy(bytes(op_c))
fr = ict.Frames(NF, 640, 480, 3, 8); fr.upload(0, np.stack(frames))
tr = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
tr.set_sum_order(int(os.environ.get('SUM_ORDER', 0)))
if os.environ.get('SEQ_LAUNCHES') == '1':
    tr.set_knob("seq_launches", 1)   # one launch per frame step instead of the whole chain in one K2v8 launch
pts = np.concatenate([sc.points(100 + s, NP, 8, 3) for s in range(S)])
tr.set_points(np.arange(S + 1, dtype=np.int64) * NP, pts)
for rep in range(3):
    t0 = time.perf_counter()
    out = tr.track_sequence(fr, 0, NF - 1, 1, np.zeros((S, 6)))
    dt = time.perf_counter() - t0
    npix = int(out["npixres"].sum())
    err = np.abs(out["poses"][-1, 0] - poses[-1]).max()
    print("frames %d samples %d: %.2f ms (%.1f us per frame step), %.3e pixel-residuals/s, %.0f tracks/s, drift vs gt %.2e"
          % (NF, S, 1e3 * dt, 1e6 * dt / (NF - 1), npix / dt, S * (NF - 1) / dt, err))
