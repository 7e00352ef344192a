"""Mixed tracking batches against the CPU oracle: uneven point counts in one batch (zero and one point included),
per-track (ref, new) frame pairs over a store of five frames, initial poses that move points out of the frame, and
every way a frame can enter the store.

The tracking kernel and its launch form are chosen from the LARGEST track of a batch (select_track_kernel), so a small
track that shares a batch with a large one runs in a form it never runs in alone; each case below pins the kernel it
exists to cover (kernels_of), so that a later routing change cannot move it off that kernel unnoticed.  Every case is
checked in the four summation orders:
  * orders 1 and 3 bit-identical to the oracle in its sum modes 0 and 1 (trace, counts, poses, reprojection);
  * orders 0 and 2 (tree sums) within 1e-5 of the oracle's first-iteration J^T r, with the same visible-point counts,
    and bit-identical to themselves on a seeded permutation of the tracks (same T and largest track, so the same
    kernel and launch form)."""
import numpy as np
import pytest

from invcompcamtrack_b200 import synth
from oracle import oracle as O
from test_gpu_kernel_routing import kernels_of, assert_routed, MULTI

pytestmark = pytest.mark.gpu

FAST, SSE, GENERAL, AVX = 0, 1, 2, 3
NFR = 5                  # frames per store
TC = 40                  # trace records per track (levels x maxiter at most 4 x 8 = 32)

_stores = {}


def store(ict, orc, psz, w, h, lv_f):
    """Five frames of a smooth camera walk, uploaded once per geometry, with the oracle's pyramids of the frames."""
    key = (psz, w, h, lv_f)
    if key not in _stores:
        sc, frames, _ = synth.make_sequence(40 + psz, NFR, w, h)
        fr = ict.Frames(NFR, w, h, lv_f, psz)
        fr.upload(0, np.stack(frames))
        pyr = [orc.pyramid_build(f.astype(np.float32), lv_f, psz) for f in frames]
        _stores[key] = dict(sc=sc, frames=frames, fr=fr, pyr=pyr, psz=psz, w=w, h=h, lv_f=lv_f)
    return _stores[key]


PAIR_KINDS = ((0, 1), (1, 0), (0, 2), (0, 0))   # forward, backward, skipping a frame, ref == new


def make_mixed(ict, st, sizes, seed, maxiter=8, ratio=0.01, lv_l=0, maxpttrack=None, donorm=0, dopatchnorm=0,
               pairs=None, dense=None):
    """Per-track point counts `sizes`, seeded points, (ref, new) pairs and initial poses; two tracks in five start
    from a pose that moves part or nearly all of their points out of the frame.  dense: index of a track that holds
    one point per pixel inside a border of 40 (psz 1)."""
    sc, psz, lv_f = st["sc"], st["psz"], st["lv_f"]
    rng = np.random.default_rng(seed)
    sizes = list(sizes)
    pts = []
    for t, n in enumerate(sizes):
        if dense is not None and t == dense:
            p = sc.dense_points(40)
            sizes[t] = p.size // 3
        else:
            p = sc.points(seed * 1000 + t, n, psz, lv_f)
        pts.append(p)
    T = len(sizes)
    pt_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    if pairs is None:
        pairs = []
        for t in range(T):
            a, b = PAIR_KINDS[t % len(PAIR_KINDS)]
            k = int(rng.integers(0, NFR - 2))
            pairs.append((k + a, k + b) if t % 2 == 0 else (NFR - 1 - k - a, NFR - 1 - k - b))
    pairs = np.array(pairs, np.int32)
    p_in = np.concatenate([rng.uniform(-0.01, 0.01, (T, 3)), rng.uniform(-0.002, 0.002, (T, 3))], 1)
    p_in[3::5, 0] += 1.0                     # pans at depth 5: part of the points leave the frame ...
    p_in[4::5, 1] += 2.5                     # ... or nearly all of them
    op = ict.make_optparam(lv_f=lv_f, lv_l=lv_l, psz=psz, maxiter=maxiter, normdp_ratio=ratio, donorm=donorm,
                           dopatchnorm=dopatchnorm, maxpttrack=maxpttrack or max(max(sizes), 1))
    return dict(st=st, op=op, sizes=sizes, pts=np.concatenate(pts), pt_off=pt_off, rf=pairs[:, 0].copy(),
                nf=pairs[:, 1].copy(), p_in=p_in, T=T)


def permuted(c, perm):
    """The same tracks in the order perm (new track j = old track perm[j])."""
    segs = [c["pts"][3 * c["pt_off"][t]:3 * c["pt_off"][t + 1]] for t in range(c["T"])]
    sizes = [c["sizes"][t] for t in perm]
    d = dict(c)
    d.update(sizes=sizes, pts=np.concatenate([segs[t] for t in perm]),
             pt_off=np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64), rf=c["rf"][perm].copy(),
             nf=c["nf"][perm].copy(), p_in=c["p_in"][perm].copy())
    return d


def pt2d_segments(pt2d, pt_off):
    return [pt2d[2 * pt_off[t]:2 * pt_off[t + 1]] for t in range(len(pt_off) - 1)]


def oracle_mixed(orc, c, sum_mode=0):
    st = c["st"]
    op = O.OptParam.from_buffer_copy(bytes(c["op"]))
    orc.set_sum_mode(sum_mode)
    try:
        return orc.track_batch(op, st["sc"].fc, st["sc"].cc, st["sc"].wh, [q[0] for q in st["pyr"]],
                               [q[1] for q in st["pyr"]], [q[2] for q in st["pyr"]], c["pt_off"], c["pts"].copy(),
                               c["rf"], c["nf"], c["p_in"], trace_cap=TC, nthreads=0, want_pt2d=True)
    finally:
        orc.set_sum_mode(0)


def new_tracker(ict, c, order, knobs=()):
    sc = c["st"]["sc"]
    tr = ict.Tracker(ict.OptParam.from_buffer_copy(bytes(c["op"])), sc.fc, sc.cc, sc.wh)
    tr.set_sum_order(order)
    for k, v in knobs:
        tr.set_knob(k, v)
    tr.set_points(c["pt_off"], c["pts"].copy())
    return tr


def gpu_mixed(ict, c, order, knobs=(), fr=None, profile=False):
    """One track_batch call; with profile, also the names of the kernels it launched."""
    tr = new_tracker(ict, c, order, knobs)
    fr = fr or c["st"]["fr"]
    out = {}
    try:
        call = lambda: out.update(tr.track_batch(fr, c["rf"], c["nf"], c["p_in"], trace_cap=TC))   # noqa: E731
        names = kernels_of(call) if profile else call()
        out["pt2d"] = tr.get_2dpoints()
        out["kernels"] = names
    finally:
        tr.close()
    return out


def assert_same(g, o):
    """Every output EQUAL; NaN where the other side has NaN (degenerate donorm tracks)."""
    assert np.array_equal(g["iters"], o["iters"]), (g["iters"], o["iters"])
    assert np.array_equal(g["npixres"], o["npixres"])
    assert np.array_equal(g["trace"][..., :16], o["trace"][..., :16], equal_nan=True), \
        "per-iteration trace (level, it, J^T r, delta_p, normdp, nvis)"
    assert np.array_equal(g["p_out"], o["p_out"], equal_nan=True)
    assert np.array_equal(g["pt2d"], o["pt2d"], equal_nan=True)


def assert_close_first_iteration(g, o, c):
    """Tree-order kernels: J^T r of each track's first iteration (identical inputs) within 1e-5 of sum|sd * r|, the
    same number of visible points there; degenerate (NaN) tracks NaN in the same places, J^T r exactly 0 where no point
    is visible.  A track with ref == new has a residual of exactly 0 in the reference order, so sum|sd * r| is 0 and
    there is no scale for the tree-order kernels, which sample the new frame with a fused bilinear formula (its
    rounding differs from the template's): those tracks are checked bit for bit in orders 1 and 3 only."""
    assert np.array_equal(g["trace"][:, 0, 15], o["trace"][:, 0, 15])
    for t in range(c["T"]):
        if np.isnan(o["p_out"][t]).any():
            assert np.array_equal(g["p_out"][t], o["p_out"][t], equal_nan=True), t
            continue
        if o["trace"][t, 0, 15] == 0:
            assert (g["trace"][t, 0, 2:8] == 0).all(), (t, g["trace"][t, 0, 2:8])
            continue
        if c["rf"][t] == c["nf"][t]:
            continue
        scale = np.maximum(o["trace"][t, 0, 16:22].astype(np.float64), 1e-30)
        d = np.abs(g["trace"][t, 0, 2:8].astype(np.float64) - o["trace"][t, 0, 2:8]) / scale
        assert d.max() <= 1e-5, (t, c["sizes"][t], d)


def assert_equal_runs(g, r, what=""):
    """Two GPU runs of the same tracks: the same bits (trace records without their cycle counts, 16-23)."""
    for k in ("p_out", "iters", "npixres", "trace", "pt2d"):
        if k in g and k in r:
            a, b = (g[k][..., :16], r[k][..., :16]) if k == "trace" else (g[k], r[k])
            assert np.array_equal(a, b, equal_nan=True), (what, k)


def assert_permutation_invariant(g, gp, perm, c, cp):
    """gp ran the tracks of g in the order perm: every output of a track must be the same bits."""
    assert_equal_runs(gp, {k: g[k][perm] for k in ("p_out", "iters", "npixres", "trace")}, "permuted")
    a, b = pt2d_segments(g["pt2d"], c["pt_off"]), pt2d_segments(gp["pt2d"], cp["pt_off"])
    for j, t in enumerate(perm):
        assert np.array_equal(b[j], a[t], equal_nan=True), (j, t)


def check_routed(names, want):
    if isinstance(want, tuple):                   # the multi-CTA path with these fused dense kernels among its launches
        assert all(n.startswith(("k_big_", "k_dense_")) for n in names), sorted(set(names))
        assert set(want) <= set(names), sorted(set(names))
    else:
        assert_routed(names, want)


def family(want):
    """TrackKernel (select_track_kernel) of a kernel name."""
    if isinstance(want, tuple) or want == MULTI:
        return "MultiCta"
    if want == "k_track_x":
        return "X"
    return {"k_track_v8": "V8", "k_track_v2": "V2", "k_track_fast": "Fast", "k_track_x8": "X8", "k_track_r": "R",
            "k_track": "General"}[want.split("<")[0]]


# psz, geometry, sizes, builder options, kernel per order {0, 1, 2, 3}
G8 = (8, 640, 480, 3)
G16 = (16, 960, 544, 3)
G32 = (32, 1280, 704, 3)
G32_NO_TMA = (32, 1288, 728, 3)    # padded rows of levels 2 and 3 not a multiple of 16 bytes: no tensor maps
DENSE = ("k_dense_iter_tma<3>", "k_dense_iter")   # fast mode, psz 1: bulk-copy form for track 0, plain loads after it

MIXED = [
    pytest.param(G8, [0, 1, 3, 13, 64, 100, 128], {},
                 {FAST: "k_track_v8<false,true,8>", SSE: "k_track_x8<false,15,1,4>", GENERAL: "k_track<8,0>",
                  AVX: "k_track_x8<false,15,1,8>"}, id="psz8-v8w8"),
    pytest.param(G8, [1, 7, 129, 150, 190], dict(dopatchnorm=1),
                 {FAST: "k_track_v8<true,true,16>", SSE: "k_track_x8<true,15,1,4>", GENERAL: "k_track<8,1>",
                  AVX: "k_track_x8<true,15,1,8>"}, id="psz8-v8w16-patchnorm"),
    pytest.param(G8, [1, 7, 129, 150, 190, 1], dict(donorm=1),
                 {FAST: "k_track_v8<false,true,16>", SSE: "k_track_x8<false,15,1,4>", GENERAL: "k_track<8,0>",
                  AVX: "k_track_x8<false,15,1,8>"}, id="psz8-v8w16-donorm"),
    pytest.param(G8, [int(n) for n in np.random.default_rng(5).integers(1, 101, 170)], dict(maxiter=4),
                 {FAST: "k_track_v8<false,true,8>", SSE: "k_track_x8<false,7,1,4>", GENERAL: "k_track<8,0>",
                  AVX: "k_track_x8<false,7,1,8>"}, id="psz8-170tracks-x8np7"),
    pytest.param(G8, [5, 90, 17, 41, 40, 88, 6], dict(maxpttrack=40),
                 {FAST: "k_track_v8<false,true,8>", SSE: "k_track_x8<false,15,1,4>", GENERAL: "k_track<8,0>",
                  AVX: "k_track_x8<false,15,1,8>"}, id="psz8-cap40"),
    pytest.param(G16, [0, 1, 9, 17, 40], {},
                 {FAST: "k_track_fast<16,4,4>", SSE: "k_track_x8<false,15,4,4>", GENERAL: "k_track<16,0>",
                  AVX: "k_track_x8<false,15,4,8>"}, id="psz16"),
    pytest.param(G32, [0, 1, 2, 4, 1, 4], {},
                 {FAST: "k_track_v2<16,4,true,256>", SSE: "k_track_r<4,2>", GENERAL: "k_track<32,0>",
                  AVX: "k_track<32,6>"}, id="psz32-k2r4"),
    pytest.param(G32, [1, 3, 5, 8, 0, 8], {},
                 {FAST: "k_track_v2<16,2,true,512>", SSE: "k_track_r<8,2>", GENERAL: "k_track<32,0>",
                  AVX: "k_track<32,6>"}, id="psz32-k2r8"),
    pytest.param(G32, [1, 4, 9, 13, 0], {},
                 {FAST: "k_track_v2<16,1,true,1024>", SSE: "k_track_x", GENERAL: "k_track<32,0>",
                  AVX: "k_track<32,6>"}, id="psz32-v2-k2x"),
    pytest.param(G32_NO_TMA, [1, 4, 8, 0], {},
                 {FAST: "k_track_v2<16,2,true,512>", SSE: "k_track_x", GENERAL: "k_track<32,0>",
                  AVX: "k_track<32,6>"}, id="psz32-no-tensor-maps"),
    pytest.param((4, 640, 480, 3), [0, 1, 5, 50], {},
                 {FAST: "k_track<0,0>", SSE: "k_track<0,2>", GENERAL: "k_track<0,0>", AVX: "k_track<0,6>"}, id="psz4"),
    pytest.param((7, 640, 480, 3), [0, 1, 5, 50], dict(dopatchnorm=1),
                 {FAST: "k_track<0,1>", SSE: "k_track<0,3>", GENERAL: "k_track<0,1>", AVX: "k_track<0,7>"},
                 id="psz7-patchnorm"),
    pytest.param(G8, [300, 1, 0, 250], dict(maxiter=5),
                 {FAST: MULTI, SSE: MULTI, GENERAL: MULTI, AVX: MULTI}, id="psz8-multi-cta"),
    pytest.param((1, 320, 240, 2), [0, 8], dict(dense=0, maxiter=6),
                 {FAST: DENSE, SSE: MULTI, GENERAL: MULTI, AVX: MULTI}, id="dense-first"),
    pytest.param((1, 320, 240, 2), [8, 0], dict(dense=1, maxiter=6),
                 {FAST: DENSE, SSE: MULTI, GENERAL: MULTI, AVX: MULTI}, id="dense-second"),
]


@pytest.mark.parametrize("geom,sizes,kw,want", MIXED)
def test_mixed_batch(ict, orc, geom, sizes, kw, want):
    st = store(ict, orc, *geom)
    c = make_mixed(ict, st, sizes, seed=sum(sizes) % 1000 + len(sizes), **kw)
    if c["T"] >= 4:
        assert len(set(c["rf"].tolist() + c["nf"].tolist())) >= 3 and (c["rf"] == c["nf"]).any()
    o0, o1 = oracle_mixed(orc, c, 0), oracle_mixed(orc, c, 1)
    perm = np.random.default_rng(c["T"]).permutation(c["T"])
    if (perm == np.arange(c["T"])).all():
        perm = np.roll(perm, 1)
    cp = permuted(c, perm)
    for order in (SSE, AVX, FAST, GENERAL):
        g = gpu_mixed(ict, c, order, profile=True)
        check_routed(g["kernels"], want[order])
        if order in (SSE, AVX):
            assert_same(g, o0 if order == SSE else o1)
        else:
            assert_close_first_iteration(g, o0, c)
            assert_permutation_invariant(g, gpu_mixed(ict, cp, order), perm, c, cp)
    if geom[0] == 32 and want[SSE].startswith("k_track_r"):
        # the same bits from K2x: knob no_k2r
        g = gpu_mixed(ict, c, SSE, knobs=(("no_k2r", 1),), profile=True)
        assert_routed(g["kernels"], "k_track_x")
        assert_same(g, o0)


def test_every_kernel_family_is_pinned():
    """Each TrackKernel (V8, V2, Fast, X8, R, X, General, MultiCta) is the kernel of at least one mixed case."""
    pinned = {family(w) for p in MIXED for w in p.values[3].values()}
    assert pinned == {"V8", "V2", "Fast", "X8", "R", "X", "General", "MultiCta"}


# ---- ict_track_sequence on uneven tracks -----------------------------------------------------------------------------
def test_sequence_uneven_tracks(ict, orc):
    """Forward over the five frames and back: order 1 equals an oracle chain step by step; in the fast mode the
    one-launch K2v8 chain equals one launch per step (seq_launches) bit for bit."""
    st = store(ict, orc, *G8)
    sizes = [0, 1, 3, 13, 64, 100]
    c = make_mixed(ict, st, sizes, seed=61, maxiter=6)
    for first, step in ((0, 1), (NFR - 1, -1)):
        tr = new_tracker(ict, c, SSE)
        g = tr.track_sequence(st["fr"], first, NFR - 1, step, c["p_in"])
        tr.close()
        p = c["p_in"].copy()
        assert np.array_equal(g["poses"][0], p)
        for k in range(NFR - 1):
            fr_k = first + k * step
            ck = dict(c, rf=np.full(c["T"], fr_k, np.int32), nf=np.full(c["T"], fr_k + step, np.int32), p_in=p)
            o = oracle_mixed(orc, ck, 0)
            assert np.array_equal(g["iters"][k], o["iters"]), k
            assert np.array_equal(g["npixres"][k], o["npixres"]), k
            assert np.array_equal(g["poses"][k + 1], o["p_out"]), k
            p = o["p_out"]
        runs = []
        for seq_launches in (0, 1):
            tr = new_tracker(ict, c, FAST, knobs=(("seq_launches", seq_launches),))
            res = {}
            names = kernels_of(lambda: res.update(tr.track_sequence(st["fr"], first, NFR - 1, step, c["p_in"])))
            tr.close()
            assert names == ["k_track_v8<false,false,8>"] * (1 + (NFR - 2) * seq_launches), names
            runs.append(res)
        for k in ("poses", "iters", "npixres"):
            assert np.array_equal(runs[0][k], runs[1][k]), k


# ---- every way a frame enters the store ------------------------------------------------------------------------------
def test_frame_entry_points(ict, orc):
    """upload_planes (the oracle's pyramids; intensity only for a frame used only as a new image), build_dev and
    build_dev_u8 from device tensors on a side stream: the stored planes equal the uploaded store's bit for bit, and
    tracking a mixed batch on each store equals tracking on the uploaded one."""
    import torch
    st = store(ict, orc, *G8)
    w, h, lv_f, psz = st["w"], st["h"], st["lv_f"], st["psz"]
    sizes = [0, 1, 7, 40, 100, 3]
    pairs = [(0, 1), (1, 0), (0, 2), (2, 2), (3, 4), (2, 4)]   # frame 4 is only ever the new image
    c = make_mixed(ict, st, sizes, seed=71, pairs=pairs, maxiter=6)
    ref = {o: gpu_mixed(ict, c, o) for o in (SSE, FAST)}
    assert_same(ref[SSE], oracle_mixed(orc, c, 0))
    up = [st["fr"].download(f) for f in range(NFR)]

    planes = ict.Frames(NFR, w, h, lv_f, psz)
    for f in range(NFR - 1):
        planes.upload_planes(f, *st["pyr"][f])
    planes.upload_planes(NFR - 1, st["pyr"][NFR - 1][0])
    imgs = np.stack(st["frames"])
    side = torch.cuda.Stream()
    built = {}
    for name, dt in (("dev_f32", torch.float32), ("dev_u8", torch.uint8)):
        t = torch.from_numpy(imgs).to(dtype=dt).cuda()
        torch.cuda.synchronize()
        fr = ict.Frames(NFR, w, h, lv_f, psz)
        fr.build_dev(0, NFR, t.data_ptr(), u8=dt == torch.uint8, stream=side.cuda_stream)
        side.synchronize()
        built[name] = (fr, t)
    stores = dict(planes=planes, **{k: v[0] for k, v in built.items()})
    try:
        for name, fr in stores.items():
            for f in range(NFR):
                got = fr.download(f)
                n = 1 if (name == "planes" and f == NFR - 1) else 3
                for k in range(n):
                    assert np.array_equal(got[k], up[f][k]), (name, f, k)
            for o in (SSE, FAST):
                assert_equal_runs(gpu_mixed(ict, c, o, fr=fr), ref[o], (name, o))
    finally:
        for fr in stores.values():
            fr.close()


@pytest.mark.parametrize("geom,sizes,order,want", [(G32, [1, 4, 0, 2, 3, 4], SSE, "k_track_r<4,2>"),
                                                   (G8, [0, 1, 13, 64, 100, 5], FAST, "k_track_v8<false,true,8>")])
def test_view_store_aliases(ict, orc, geom, sizes, order, want):
    """A view whose entries alias the frames of two owning stores in shuffled order tracks bit-identically to the same
    pairs on one owning store (with psz 32 the tensor maps travel with the frame descriptor)."""
    st = store(ict, orc, *geom)
    psz, w, h, lv_f = geom
    c = make_mixed(ict, st, sizes, seed=81, maxiter=6)
    ref = gpu_mixed(ict, c, order)
    other = ict.Frames(NFR, w, h, lv_f, psz)
    other.upload(0, np.stack(st["frames"]))
    view = ict.Frames(NFR, w, h, lv_f, psz, view=True)
    rng = np.random.default_rng(82)
    where = rng.permutation(NFR)                  # view entry where[f] holds frame f
    for f in range(NFR):
        src = other if f % 2 else st["fr"]
        view.alias(int(where[f]), src, f)
    try:
        cv = dict(c, rf=where[c["rf"]].astype(np.int32), nf=where[c["nf"]].astype(np.int32))
        g = gpu_mixed(ict, cv, order, fr=view, profile=True)
        assert_routed(g["kernels"], want)
        assert_equal_runs(g, ref)
    finally:
        view.close()
        other.close()


@pytest.mark.parametrize("geom,sizes,order", [(G8, [0, 1, 13, 64, 100, 5], SSE), (G8, [0, 1, 13, 64, 100, 5], FAST),
                                              (G32, [1, 4, 0, 2], SSE), (G8, [300, 1, 0], SSE)])
def test_track_batch_dev(ict, orc, geom, sizes, order):
    """ict_track_batch_dev with device arrays equals ict_track_batch; the multi-CTA path refuses it."""
    import torch
    st = store(ict, orc, *geom)
    c = make_mixed(ict, st, sizes, seed=91, maxiter=6)
    T, L = c["T"], c["op"].lv_f - c["op"].lv_l + 1
    tr = new_tracker(ict, c, order)
    try:
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()   # noqa: E731
        rf, nf, p_in = dev(c["rf"]), dev(c["nf"]), dev(c["p_in"])
        p_out = torch.zeros((T, 6), dtype=torch.float64, device="cuda")
        iters = torch.zeros((T, L), dtype=torch.int32, device="cuda")
        npix = torch.zeros(T, dtype=torch.int64, device="cuda")
        trace = torch.zeros((T, TC, 24), dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()
        call = lambda: tr.track_batch_dev(st["fr"], rf.data_ptr(), nf.data_ptr(), p_in.data_ptr(),   # noqa: E731
                                          p_out.data_ptr(), iters.data_ptr(), npix.data_ptr(), trace.data_ptr(), TC)
        if max(sizes) >= 300:
            with pytest.raises(ict.IctError, match="ICT_ERR_UNSUPPORTED"):
                call()
            return
        call()
        torch.cuda.synchronize()
        ref = tr.track_batch(st["fr"], c["rf"], c["nf"], c["p_in"], trace_cap=TC)
    finally:
        tr.close()
    assert_equal_runs(dict(p_out=p_out.cpu().numpy(), iters=iters.cpu().numpy(), npixres=npix.cpu().numpy(),
                           trace=trace.cpu().numpy()), ref)


def test_reproject_uneven_tracks_with_cap(ict, orc):
    """ict_tracker_reproject on uneven tracks with a maxpttrack cap equals the oracle's reference reprojection (zeros
    beyond the cap), and again on the same tracker after set_points with a smaller layout."""
    st = store(ict, orc, *G8)
    c = make_mixed(ict, st, [5, 90, 0, 41, 1, 60], seed=101, maxpttrack=40, maxiter=1)
    tr = new_tracker(ict, c, SSE)
    try:
        q = tr.reproject(c["p_in"])
        assert np.array_equal(q, oracle_mixed(orc, c)["pt2d"])
        segs = pt2d_segments(q, c["pt_off"])
        for t, n in enumerate(c["sizes"]):
            if n > 40:
                assert (segs[t][40:n] == 0).all() and (segs[t][n + 40:] == 0).all()
        small = make_mixed(ict, st, [3, 0, 12], seed=102, maxpttrack=40, maxiter=1)
        tr.set_points(small["pt_off"], small["pts"].copy())
        assert np.array_equal(tr.reproject(small["p_in"]), oracle_mixed(orc, small)["pt2d"])
    finally:
        tr.close()


# ---- ict_tracker_set_optparam ----------------------------------------------------------------------------------------
def test_set_optparam_between_calls(ict, orc):
    """lv_l, maxiter, normdp_ratio and dopatchnorm may change between calls: each call gives the bits of a fresh
    tracker with the new optparam (orders 0 and 1)."""
    st = store(ict, orc, *G8)
    c = make_mixed(ict, st, [0, 1, 13, 64, 100, 5], seed=111, maxiter=6)
    M = c["op"].maxpttrack
    ops = [dict(lv_l=1), dict(maxiter=3, normdp_ratio=0.05), dict(dopatchnorm=1), {}]
    for order in (FAST, SSE):
        tr = new_tracker(ict, c, order)
        try:
            for kw in ops:
                a = dict(lv_f=3, lv_l=0, psz=8, maxiter=6, normdp_ratio=0.01, dopatchnorm=0, maxpttrack=M)
                a.update(kw)
                op = ict.make_optparam(**a)
                tr.set_optparam(op)
                g = tr.track_batch(st["fr"], c["rf"], c["nf"], c["p_in"], trace_cap=TC)
                assert_equal_runs(g, gpu_mixed(ict, dict(c, op=op), order), (order, kw))
        finally:
            tr.close()


@pytest.mark.parametrize("change", [dict(maxpttrack=200), dict(maxpttrack=40), dict(donorm=1)])
def test_set_optparam_refuses_stale_points(ict, orc, change):
    """A maxpttrack or donorm other than the one the points were stored with: every call that reads the points is
    refused until set_points runs again; then the tracker equals a fresh one."""
    st = store(ict, orc, *G8)
    c = make_mixed(ict, st, [0, 1, 13, 64, 100, 5], seed=121, maxiter=6)
    tr = new_tracker(ict, c, SSE)
    try:
        tr.track_batch(st["fr"], c["rf"], c["nf"], c["p_in"])
        a = dict(lv_f=3, psz=8, maxiter=6, maxpttrack=c["op"].maxpttrack)
        a.update(change)
        op = ict.make_optparam(**a)
        tr.set_optparam(op)
        for call in (lambda: tr.track_batch(st["fr"], c["rf"], c["nf"], c["p_in"]),
                     lambda: tr.track_sequence(st["fr"], 0, 2, 1, c["p_in"]),
                     lambda: tr.reproject(c["p_in"]), tr.get_2dpoints):
            with pytest.raises(ict.IctError, match="ICT_ERR_BAD_ARG.*set_points"):
                call()
        tr.set_points(c["pt_off"], c["pts"].copy())
        g = tr.track_batch(st["fr"], c["rf"], c["nf"], c["p_in"], trace_cap=TC)
        g["pt2d"] = tr.get_2dpoints()
    finally:
        tr.close()
    c2 = dict(c, op=op)
    assert_equal_runs(g, gpu_mixed(ict, c2, SSE))
    assert_same(g, oracle_mixed(orc, c2))
