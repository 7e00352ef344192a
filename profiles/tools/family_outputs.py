"""Outputs of every tracking kernel family on fixed seeded inputs, for comparing two builds bit for bit.

    python profiles/tools/family_outputs.py OUT_DIR            # writes OUT_DIR/<case>.npz
    python profiles/tools/family_outputs.py --compare DIR_A DIR_B

Each case pins one kernel family and template instance (the rows of tests/test_gpu_kernel_routing.py) and runs a
three-track batch with uneven point counts and a trace; it saves p_out, iters, npixres, trace[..., :16] and
get_2dpoints().  The K2v8 case with a frame chain runs ict_track_sequence in one launch, and one case runs reproject.
The kernels are deterministic, so two runs of the same build give identical files."""
import os
import sys

import numpy as np

R = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, R)

FAST, SSE, GENERAL, AVX = 0, 1, 2, 3
GEOM = {1: (320, 240, 2), 4: (640, 480, 3), 8: (640, 480, 3), 16: (960, 544, 3), 32: (1920, 1080, 3)}
# name: psz, points of the largest track, sum order, dopatchnorm, tracks
CASES = {
    "v8_p100": (8, 100, FAST, 0, 3), "v8_pn": (8, 50, FAST, 1, 3), "v8_nw16": (8, 200, FAST, 0, 3),
    "v2_p4": (32, 4, FAST, 0, 3), "v2_p8": (32, 8, FAST, 0, 3), "v2_p17": (32, 17, FAST, 0, 3),
    "fast_psz8": (8, 250, FAST, 0, 3), "fast_psz16": (16, 70, FAST, 0, 3), "fast_psz32": (32, 18, FAST, 0, 3),
    "x8_np15": (8, 100, SSE, 0, 3), "x8_np7": (8, 24, SSE, 0, 170), "x8_pn": (8, 50, SSE, 1, 3),
    "x8_psz16": (16, 55, SSE, 0, 3), "x8_avx": (8, 100, AVX, 0, 3),
    "r_p4": (32, 4, SSE, 0, 3), "r_p8": (32, 8, SSE, 0, 3), "x_p13": (32, 13, SSE, 0, 3),
    "general_o0": (4, 50, FAST, 0, 3), "general_o1": (4, 50, SSE, 1, 3), "general_o2": (8, 100, GENERAL, 0, 3),
    "general_o3": (4, 50, AVX, 0, 3), "general_pn32": (32, 13, FAST, 1, 3),
    "multi_psz1": (1, 3000, FAST, 0, 1), "multi_psz1_sse": (1, 3000, SSE, 0, 1), "multi_psz8": (8, 261, FAST, 0, 2),
}
TRACE_CAP = 64


def setup(ict, synth, psz, npts, order, pn, ntracks, nframes=2):
    w, h, lv_f = GEOM[psz]
    sc, A, B, _ = synth.make_pair(5, w, h)
    fr = ict.Frames(nframes, w, h, lv_f, psz)
    fr.upload(0, np.stack([A, B] * (nframes // 2)))
    op = ict.make_optparam(lv_f=lv_f, psz=psz, maxiter=10, dopatchnorm=pn, maxpttrack=npts)
    tr = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
    tr.set_sum_order(order)
    counts = [max(1, npts - (k % 3) * (npts // 3)) for k in range(ntracks)]   # uneven: n, 2n/3, n/3, n, ...
    pts = np.concatenate([sc.points(11 + t, n, psz, lv_f) for t, n in enumerate(counts)])
    tr.set_points(np.concatenate([[0], np.cumsum(counts)]).astype(np.int64), pts)
    p_in = np.zeros((ntracks, 6))
    p_in[:, 0] = 1e-3 * np.arange(ntracks)
    return tr, fr, p_in


def run(out_dir):
    import invcompcamtrack_b200 as ict
    from invcompcamtrack_b200 import synth
    os.makedirs(out_dir, exist_ok=True)
    for name, (psz, npts, order, pn, ntracks) in CASES.items():
        tr, fr, p_in = setup(ict, synth, psz, npts, order, pn, ntracks)
        try:
            out = tr.track_batch(fr, 0, 1, p_in, trace_cap=TRACE_CAP)
            np.savez(os.path.join(out_dir, name + ".npz"), p_out=out["p_out"], iters=out["iters"],
                     npixres=out["npixres"], trace=out["trace"][..., :16], pt2d=tr.get_2dpoints())
            if name == "v8_p100":
                np.savez(os.path.join(out_dir, "reproject.npz"), pt2d=tr.reproject(p_in + 1e-3))
        finally:
            tr.close()
    tr, fr, p_in = setup(ict, synth, 8, 100, FAST, 0, 3, nframes=4)   # K2v8's one-launch frame chain
    try:
        out = tr.track_sequence(fr, 0, 3, 1, p_in)
        np.savez(os.path.join(out_dir, "v8_seq.npz"), **out)
    finally:
        tr.close()
    print("wrote", len(os.listdir(out_dir)), "files to", out_dir)


def compare(a, b):
    bad = 0
    names = sorted(os.listdir(a))
    assert names == sorted(os.listdir(b)), (names, sorted(os.listdir(b)))
    for n in names:
        x, y = np.load(os.path.join(a, n)), np.load(os.path.join(b, n))
        for k in x.files:
            same = np.array_equal(x[k], y[k], equal_nan=x[k].dtype.kind == "f")
            bad += not same
            if not same:
                print("DIFFERENT", n, k)
    print("%d files, %s" % (len(names), "all arrays identical" if not bad else "%d arrays differ" % bad))
    return bad


if __name__ == "__main__":
    if sys.argv[1] == "--compare":
        sys.exit(1 if compare(sys.argv[2], sys.argv[3]) else 0)
    run(sys.argv[1])
