"""Which tracking kernel runs for each configuration (select_track_kernel, csrc/ict_kernels.cu).

Every reference-order kernel is bit-identical to the oracle and to the others, and the fast-mode kernels agree within
summation noise, so a track sent to the wrong kernel passes every parity test and only runs at another speed.  These
cases pin the choice itself: each runs one small tracking call under torch.profiler and compares the names of the
kernels it launched, template arguments included, with the table in DESIGN.md §4.  The boundary rows follow from the
shared-memory sizing of each kernel (224 256 bytes per CTA at most)."""
import re

import numpy as np
import pytest

from invcompcamtrack_b200 import synth

FAST, SSE, GENERAL, AVX = 0, 1, 2, 3          # ict_tracker_set_sum_order
MULTI = "multi-CTA"                           # k_big_* launches only
DENSE_TMA = "dense: k_dense_iter_tma<3>"      # multi-CTA path with the fused dense iteration, bulk-copy form
DENSE_LDG = "dense: k_dense_iter"             # ... and its form for unaligned point counts

GEOM = {1: (320, 240, 2), 4: (640, 480, 3), 8: (640, 480, 3), 16: (960, 544, 3), 32: (1920, 1080, 3)}
NO_TMA = (1288, 728, 3)   # psz 32 without tensor maps: padded level-2 and level-3 rows are not multiples of 16 bytes

_frames = {}


def frames(ict, psz, geom, nframes=2):
    """A frame store of the synthetic pair (A, B, A, B, ...) for this patch size and geometry, shared by the cases."""
    key = (psz, geom, nframes)
    if key not in _frames:
        w, h, lv_f = geom
        sc, A, B, _ = synth.make_pair(5, w, h)
        fr = ict.Frames(nframes, w, h, lv_f, psz)
        fr.upload(0, np.stack([A, B] * (nframes // 2)))
        _frames[key] = (sc, fr)
    return _frames[key]


def kernels_of(fn):
    """Names (without spaces) of the ict:: kernels fn launches, in launch order."""
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    names = [re.sub(r"\s+", "", e.name) for e in prof.events()]
    ours = [m.group(1) for m in (re.search(r"ict::(k_\w+(?:<[^<>]*>)?)", n) for n in names) if m]
    assert ours, "the profiler saw no ict:: kernel; it saw %s" % sorted(set(names))
    return ours


def tracker(ict, psz, npts, order, pn=0, ntracks=1, geom=None, knobs=(), robust=0, nframes=2):
    geom = geom or GEOM[psz]
    sc, fr = frames(ict, psz, geom, nframes)
    op = ict.make_optparam(lv_f=geom[2], psz=psz, maxiter=2, dopatchnorm=pn, maxpttrack=npts)
    tr = ict.Tracker(op, sc.fc, sc.cc, sc.wh)
    tr.set_sum_order(order)
    for k, v in knobs:
        tr.set_knob(k, v)
    if robust:
        tr.set_robust(robust)
    pts = np.concatenate([sc.points(11 + t, npts, psz, geom[2]) for t in range(ntracks)])
    tr.set_points(np.arange(ntracks + 1, dtype=np.int64) * npts, pts)
    return tr, fr


def routed(ict, psz, npts, order, **kw):
    tr, fr = tracker(ict, psz, npts, order, **kw)
    try:
        return kernels_of(lambda: tr.track_batch(fr, 0, 1, np.zeros(6)))
    finally:
        tr.close()


def assert_routed(names, want):
    if want in (MULTI, DENSE_TMA, DENSE_LDG):
        assert all(n.startswith(("k_big_", "k_dense_")) for n in names), sorted(set(names))
        dense = sorted({n for n in names if n.startswith("k_dense_iter")})
        assert dense == {MULTI: [], DENSE_TMA: ["k_dense_iter_tma<3>"], DENSE_LDG: ["k_dense_iter"]}[want], dense
    else:
        assert sorted(set(names)) == [want] and len(names) == 1, names


def row(psz, npts, order, want, **kw):
    return pytest.param(psz, npts, order, kw, want, id="psz%d-P%d-o%d%s" % (
        psz, npts, order, "".join("-%s%s" % (k, v if not isinstance(v, tuple) else "") for k, v in kw.items())))


ROWS = [
    # ---- order 0, fast mode ----
    row(8, 100, FAST, "k_track_v8<false,false,8>"),
    row(8, 128, FAST, "k_track_v8<false,false,8>"),
    row(8, 129, FAST, "k_track_v8<false,false,16>"),
    row(8, 241, FAST, "k_track_v8<false,false,16>"),
    row(8, 50, FAST, "k_track_v8<true,false,8>", pn=1),
    row(8, 241, FAST, "k_track_v8<true,false,16>", pn=1),
    row(8, 242, FAST, "k_track_fast<8,4,4>"),
    row(8, 260, FAST, "k_track_fast<8,4,4>"),
    row(8, 261, FAST, MULTI),
    row(8, 242, FAST, MULTI, pn=1),
    row(32, 4, FAST, "k_track_v2<16,4,false,256>"),
    row(32, 5, FAST, "k_track_v2<16,2,false,512>"),
    row(32, 8, FAST, "k_track_v2<16,2,false,512>"),
    row(32, 9, FAST, "k_track_v2<16,1,false,1024>"),
    row(32, 17, FAST, "k_track_v2<16,1,false,1024>"),
    row(32, 18, FAST, "k_track_fast<32,16,4>"),
    row(32, 19, FAST, MULTI),
    row(32, 13, FAST, "k_track<32,1>", pn=1),
    row(32, 14, FAST, MULTI, pn=1),
    row(16, 70, FAST, "k_track_fast<16,4,4>"),
    row(16, 71, FAST, MULTI),
    row(16, 53, FAST, "k_track<16,1>", pn=1),
    row(16, 54, FAST, MULTI, pn=1),
    row(4, 50, FAST, "k_track<0,0>"),
    row(4, 50, FAST, "k_track<0,1>", pn=1),
    row(1, 2156, FAST, "k_track<0,0>"),
    row(1, 3000, FAST, DENSE_TMA),
    row(1, 3001, FAST, DENSE_LDG),
    # ---- order 1, reference order with 4-float packets ----
    row(8, 100, SSE, "k_track_x8<false,15,1,4>"),
    row(8, 24, SSE, "k_track_x8<false,7,1,4>", ntracks=170),
    row(8, 222, SSE, "k_track_x8<false,7,1,4>"),
    row(8, 223, SSE, MULTI),
    row(8, 50, SSE, "k_track_x8<true,15,1,4>", pn=1),
    row(16, 55, SSE, "k_track_x8<false,15,4,4>"),
    row(16, 56, SSE, "k_track_x8<false,7,4,4>"),
    row(16, 57, SSE, MULTI),
    row(16, 53, SSE, "k_track<16,3>", pn=1),
    row(16, 54, SSE, MULTI, pn=1),
    row(32, 4, SSE, "k_track_r<4,2>"),
    row(32, 5, SSE, "k_track_r<8,2>"),
    row(32, 8, SSE, "k_track_r<8,2>"),
    row(32, 9, SSE, "k_track_x"),
    row(32, 13, SSE, "k_track_x"),
    row(32, 14, SSE, MULTI),
    row(32, 4, SSE, "k_track_x", knobs=(("no_k2r", 1),)),
    row(32, 4, SSE, "k_track_x", geom=NO_TMA),
    row(32, 13, SSE, "k_track<32,3>", pn=1),
    row(32, 14, SSE, MULTI, pn=1),
    row(4, 50, SSE, "k_track<0,2>"),
    row(4, 50, SSE, "k_track<0,3>", pn=1),
    row(1, 3000, SSE, MULTI),
    # ---- order 3, reference order with 8-float packets ----
    row(8, 100, AVX, "k_track_x8<false,15,1,8>"),
    row(8, 222, AVX, "k_track_x8<false,7,1,8>"),
    row(8, 223, AVX, MULTI),
    row(8, 50, AVX, "k_track_x8<true,15,1,8>", pn=1),
    row(16, 56, AVX, "k_track_x8<false,7,4,8>"),
    row(32, 4, AVX, "k_track<32,6>"),
    row(32, 13, AVX, "k_track<32,6>"),
    row(32, 14, AVX, MULTI),
    row(32, 4, AVX, "k_track<32,7>", pn=1),
    row(4, 50, AVX, "k_track<0,6>"),
    # ---- order 2, the general kernel forced ----
    row(8, 100, GENERAL, "k_track<8,0>"),
    row(8, 260, GENERAL, "k_track<8,0>"),
    row(8, 261, GENERAL, MULTI),
    row(8, 200, GENERAL, "k_track<8,1>", pn=1),
    row(8, 201, GENERAL, MULTI, pn=1),
    row(16, 70, GENERAL, "k_track<16,0>"),
    row(32, 18, GENERAL, "k_track<32,0>"),
    row(32, 19, GENERAL, MULTI),
    row(1, 3000, GENERAL, MULTI),
]


@pytest.mark.gpu
@pytest.mark.parametrize("psz,npts,order,kw,want", ROWS)
def test_track_batch_routing(ict, psz, npts, order, kw, want):
    assert_routed(routed(ict, psz, npts, order, **kw), want)


@pytest.mark.gpu
@pytest.mark.parametrize("order,seq_launches,want", [(FAST, 0, ["k_track_v8<false,false,8>"]),
                                                     (FAST, 1, ["k_track_v8<false,false,8>"] * 3),
                                                     (SSE, 0, ["k_track_x8<false,15,1,4>"] * 3)])
def test_sequence_launches(ict, order, seq_launches, want):
    """A 3-step ict_track_sequence: K2v8 loops over the frames in one launch unless seq_launches asks for one launch
    per step; every other kernel runs one launch per step."""
    tr, fr = tracker(ict, 8, 100, order, knobs=(("seq_launches", seq_launches),), nframes=4)
    try:
        assert kernels_of(lambda: tr.track_sequence(fr, 0, 3, 1, np.zeros(6))) == want
    finally:
        tr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("psz,npts,order,ok", [(8, 100, FAST, True), (8, 241, FAST, True), (8, 242, FAST, False),
                                               (8, 100, SSE, False), (8, 100, GENERAL, False),
                                               (32, 4, FAST, False)])
def test_robust_only_on_k2v8(ict, psz, npts, order, ok):
    tr, fr = tracker(ict, psz, npts, order, robust=1)
    try:
        if ok:
            assert kernels_of(lambda: tr.track_batch(fr, 0, 1, np.zeros(6)))[0].startswith("k_track_v8<")
        else:
            with pytest.raises(ict.IctError, match="ICT_ERR_UNSUPPORTED"):
                tr.track_batch(fr, 0, 1, np.zeros(6))
    finally:
        tr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("psz,npts,order,ok", [(8, 100, SSE, True), (8, 222, AVX, True), (8, 223, SSE, False),
                                               (16, 20, SSE, False), (8, 100, FAST, False), (8, 100, GENERAL, False),
                                               (32, 4, SSE, False)])
def test_keep_state_only_on_k2x8_psz8(ict, psz, npts, order, ok):
    tr, fr = tracker(ict, psz, npts, order, knobs=(("keep_state", 1),))
    try:
        if ok:
            assert kernels_of(lambda: tr.track_batch(fr, 0, 1, np.zeros(6)))[0].startswith("k_track_x8<")
        else:
            with pytest.raises(ict.IctError, match="ICT_ERR_UNSUPPORTED"):
                tr.track_batch(fr, 0, 1, np.zeros(6))
    finally:
        tr.close()
