"""ctypes binding of libictrack.so (include/ictrack.h).  Mirrors how the reference binds its C code
(misc_src/func_util_geom.py:582-604: LoadLibrary, argtypes, caller-allocated contiguous numpy buffers)."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TRACE_FLOATS = 24
MAX_LEVELS = 8
_ERR = {1: "ICT_ERR_NO_DEVICE", 2: "ICT_ERR_BAD_ARG", 3: "ICT_ERR_CUDA", 4: "ICT_ERR_NOMEM", 5: "ICT_ERR_UNSUPPORTED"}


ROBUST_FULL_STEP, ROBUST_COMPOSE, ROBUST_FLOOR = 1, 2, 4
# Tracker.set_sum_order (ict_tracker_set_sum_order)
SUM_ORDER_FAST, SUM_ORDER_EIGEN_SSE, SUM_ORDER_GENERAL_TREE, SUM_ORDER_EIGEN_AVX = 0, 1, 2, 3


class IctError(RuntimeError):
    pass


class OptParam(C.Structure):
    """ict_optparam == CTR::optparam (utilities.h:46-61)."""
    _fields_ = [("maxpttrack", C.c_int), ("psz", C.c_int), ("pszd2", C.c_int), ("pszd2m3", C.c_int),
                ("novals", C.c_int), ("lv_f", C.c_int), ("lv_l", C.c_int), ("donorm", C.c_ubyte),
                ("dopatchnorm", C.c_ubyte), ("maxiter", C.c_int), ("normdp_ratio", C.c_float),
                ("verbosity", C.c_int)]


def lib_path():
    return os.path.join(HERE, "libictrack.so")


_lib = None
_f = C.POINTER(C.c_float)
_d = C.POINTER(C.c_double)
_i = C.POINTER(C.c_int)
_l = C.POINTER(C.c_int64)
_u8 = C.POINTER(C.c_ubyte)

# every symbol include/ictrack.h declares: (restype, argtypes)
SIGNATURES = {
    "ict_optparam_init": (None, [C.POINTER(OptParam), C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int,
                                 C.c_int, C.c_int]),
    "ict_version": (C.c_int, []),
    "ict_last_error": (C.c_char_p, []),
    "ict_device_count": (C.c_int, []),
    "ict_set_device": (C.c_int, [C.c_int]),
    "ict_camera_levels": (C.c_int, [C.c_int, _f, _f, _i, C.c_int, _f]),
    "ict_pyramid_layout": (C.c_int64, [C.c_int, C.c_int, C.c_int, C.c_int, _l, _i, _i]),
    "ict_pyramid_build": (C.c_int, [_f, C.c_int, C.c_int, C.c_int, C.c_int, _f, _f, _f]),
    "ict_frames_create": (C.c_void_p, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "ict_frames_destroy": (None, [C.c_void_p]),
    "ict_frames_upload": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "ict_frames_upload_u8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "ict_frames_build_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "ict_frames_build_dev_u8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "ict_frames_upload_planes": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ict_frames_create_view": (C.c_void_p, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "ict_frames_alias": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "ict_frames_download": (C.c_int, [C.c_void_p, C.c_int, _f, _f, _f]),
    "ict_tracker_create": (C.c_void_p, [C.POINTER(OptParam), _f, _f, _i]),
    "ict_tracker_destroy": (None, [C.c_void_p]),
    "ict_tracker_set_optparam": (C.c_int, [C.c_void_p, C.POINTER(OptParam)]),
    "ict_tracker_set_sum_order": (C.c_int, [C.c_void_p, C.c_int]),
    "ict_tracker_set_knob": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "ict_tracker_set_teacher": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "ict_tracker_set_robust": (C.c_int, [C.c_void_p, C.c_uint]),
    "ict_tracker_set_points": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "ict_tracker_set_points_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                                             C.c_void_p]),
    "ict_track_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_int, C.c_void_p]),
    "ict_track_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "ict_frames_upload_u8_stream": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "ict_tracker_set_points_stream": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ict_track_batch_stream": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_void_p]),
    "ict_track_sequence": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p]),
    "ict_tracker_reproject": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "ict_tracker_get_2dpoints": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ict_track_evaluate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ict_track_evaluate_poses": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                           C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p]),
    "ict_track_pair": (C.c_int, [C.POINTER(OptParam), _f, _f, _i, _f, _f, _d, C.c_int, _d, _d, C.c_void_p,
                                 C.c_void_p, C.c_int]),
    "ict_pose_hypotheses": (C.c_int, [_f, _f, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_double,
                                      C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ict_get_patches": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(OptParam), C.c_int, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p]),
    "ict_ncc_score": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_void_p]),
    "ict_launch_count": (C.c_int64, [C.c_int]),
}


def lib():
    """Loads libictrack.so; raises IctError (never falls back to anything) when it has not been built."""
    global _lib
    if _lib is None:
        p = lib_path()
        if not os.path.exists(p):
            raise IctError("libictrack.so is missing: run `python -m invcompcamtrack_b200.build` "
                           "(or __graft_entry__.build()); there is no CPU fallback")
        L = C.CDLL(p)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise IctError("%s: %s" % (_ERR.get(rc, rc), lib().ict_last_error().decode()))


def _p(a):
    return C.c_void_p(a.ctypes.data) if a is not None else None


def make_optparam(lv_f=3, lv_l=0, psz=8, maxiter=10, normdp_ratio=0.01, donorm=0, dopatchnorm=0, maxpttrack=100,
                  verbosity=0):
    op = OptParam()
    lib().ict_optparam_init(C.byref(op), lv_f, lv_l, psz, maxiter, normdp_ratio, int(donorm), int(dopatchnorm),
                            maxpttrack, verbosity)
    return op


def device_count():
    return int(lib().ict_device_count())


def launch_count(reset=False):
    return int(lib().ict_launch_count(int(reset)))


def camera_levels(noscales, fc, cc, wh, padding):
    fc = np.asarray(fc, np.float32); cc = np.asarray(cc, np.float32); wh = np.asarray(wh, np.int32)
    out = np.zeros((noscales, 8), np.float32)
    _check(lib().ict_camera_levels(noscales, fc.ctypes.data_as(_f), cc.ctypes.data_as(_f), wh.ctypes.data_as(_i),
                                   padding, out.ctypes.data_as(_f)))
    return out


def pyramid_layout(w, h, lv_f, pad):
    off = np.zeros(MAX_LEVELS, np.int64); sw = np.zeros(MAX_LEVELS, np.int32); sh = np.zeros(MAX_LEVELS, np.int32)
    tot = int(lib().ict_pyramid_layout(w, h, lv_f, pad, off.ctypes.data_as(_l), sw.ctypes.data_as(_i),
                                       sh.ctypes.data_as(_i)))
    if tot < 0:
        raise IctError("ict_pyramid_layout: w,h must be positive and divisible by 2^lv_f")
    return tot, off[:lv_f + 1].tolist(), sw[:lv_f + 1].tolist(), sh[:lv_f + 1].tolist()


def pyramid_build(img, lv_f, pad):
    """util_constructpyramide on the GPU: host image in, (I, dx, dy) flat padded plane sets out."""
    img = np.ascontiguousarray(img, np.float32)
    h, w = img.shape
    tot, _, _, _ = pyramid_layout(w, h, lv_f, pad)
    I = np.empty(tot, np.float32); dx = np.empty(tot, np.float32); dy = np.empty(tot, np.float32)
    _check(lib().ict_pyramid_build(img.ctypes.data_as(_f), w, h, lv_f, pad, I.ctypes.data_as(_f),
                                   dx.ctypes.data_as(_f), dy.ctypes.data_as(_f)))
    return I, dx, dy


class Frames:
    """Device-resident pyramids of a set of frames (ict_frames)."""

    def __init__(self, nframes, w, h, lv_f, pad, view=False):
        self.nframes, self.w, self.h, self.lv_f, self.pad = nframes, w, h, lv_f, pad
        self.h_ = (lib().ict_frames_create_view if view else lib().ict_frames_create)(nframes, w, h, lv_f, pad)
        if not self.h_:
            raise IctError("ict_frames_create: " + lib().ict_last_error().decode())
        self.plane_floats = pyramid_layout(w, h, lv_f, pad)[0]

    def close(self):
        if getattr(self, "h_", None):
            lib().ict_frames_destroy(self.h_)
            self.h_ = None

    __del__ = close

    def upload(self, first, imgs):
        """imgs: [count, h, w] float32 or uint8 host array (a pinned torch tensor's numpy view works too)."""
        imgs = np.ascontiguousarray(imgs)
        if imgs.ndim == 2:
            imgs = imgs[None]
        assert imgs.shape[1:] == (self.h, self.w)
        if imgs.dtype == np.uint8:
            _check(lib().ict_frames_upload_u8(self.h_, first, imgs.shape[0], _p(imgs)))
        else:
            imgs = np.ascontiguousarray(imgs, np.float32)
            _check(lib().ict_frames_upload(self.h_, first, imgs.shape[0], _p(imgs)))

    def upload_planes(self, frame, I, dx=None, dy=None):
        """Pre-built padded plane sets (e.g. made by another implementation of util_constructpyramide)."""
        I = np.ascontiguousarray(I, np.float32)
        dx = None if dx is None else np.ascontiguousarray(dx, np.float32)
        dy = None if dy is None else np.ascontiguousarray(dy, np.float32)
        _check(lib().ict_frames_upload_planes(self.h_, frame, _p(I), _p(dx), _p(dy)))

    def alias(self, idx, src, src_idx):
        _check(lib().ict_frames_alias(self.h_, idx, src.h_, src_idx))

    def upload_ptr(self, first, count, host_ptr, u8):
        fn = lib().ict_frames_upload_u8 if u8 else lib().ict_frames_upload
        _check(fn(self.h_, first, count, C.c_void_p(host_ptr)))

    def build_dev(self, first, count, dev_ptr, u8=False, stream=0):
        fn = lib().ict_frames_build_dev_u8 if u8 else lib().ict_frames_build_dev
        _check(fn(self.h_, first, count, C.c_void_p(dev_ptr), C.c_void_p(stream)))

    def get_patches(self, frame, level, op, mids, grad=True):
        """util_getPatch (grad=False) / util_getPatch_grad: mids [n, 2] (x, y) -> (I, dx, dy) each [n, psz*psz]."""
        mids = np.ascontiguousarray(mids, np.float32).reshape(-1, 2)
        n, nv = mids.shape[0], op.psz * op.psz
        I = np.zeros((n, nv), np.float32)
        dx = np.zeros((n, nv), np.float32) if grad else None
        dy = np.zeros((n, nv), np.float32) if grad else None
        _check(lib().ict_get_patches(self.h_, frame, level, C.byref(op), n, _p(mids), _p(I), _p(dx), _p(dy)))
        return (I, dx, dy) if grad else I

    def download(self, frame):
        I = np.empty(self.plane_floats, np.float32); dx = np.empty_like(I); dy = np.empty_like(I)
        _check(lib().ict_frames_download(self.h_, frame, I.ctypes.data_as(_f), dx.ctypes.data_as(_f),
                                         dy.ctypes.data_as(_f)))
        return I, dx, dy


class Tracker:
    """Batch of independent tracks: one track == Set3Dpoints -> SetPose -> TrackPose (odometer.cpp:171-426)."""

    def __init__(self, op, fc, cc, wh):
        self.op = op
        self.fc = np.asarray(fc, np.float32); self.cc = np.asarray(cc, np.float32); self.wh = np.asarray(wh, np.int32)
        self.h_ = lib().ict_tracker_create(C.byref(op), self.fc.ctypes.data_as(_f), self.cc.ctypes.data_as(_f),
                                           self.wh.ctypes.data_as(_i))
        if not self.h_:
            raise IctError("ict_tracker_create: " + lib().ict_last_error().decode())
        self.T = 0
        self.L = op.lv_f - op.lv_l + 1

    def close(self):
        if getattr(self, "h_", None):
            lib().ict_tracker_destroy(self.h_)
            self.h_ = None

    __del__ = close

    def set_optparam(self, op):
        _check(lib().ict_tracker_set_optparam(self.h_, C.byref(op)))
        self.op = op
        self.L = op.lv_f - op.lv_l + 1

    def set_sum_order(self, mode):
        """Order of the fp32 sums (include/ictrack.h):
        1 (library default, SUM_ORDER_EIGEN_SSE): Eigen's packet order with 4-float SSE packets, bit-identical to the
          oracle in its sum mode 0;
        3 (SUM_ORDER_EIGEN_AVX): the same with 8-float AVX packets, bit-identical to the oracle in its sum mode 1 — a
          reference built with -mavx against Eigen >= 3.3;
        0 (SUM_ORDER_FAST): fast mode, fixed-order tree sums;  2: tree sums on the general kernel (tests).
        Other values raise IctError (ICT_ERR_BAD_ARG)."""
        _check(lib().ict_tracker_set_sum_order(self.h_, int(mode)))

    def set_teacher(self, poses):
        """poses: float32 [T, trace_cap, 8] (pose after each trace record + continue flag) or None; see ictrack.h."""
        if poses is None:
            _check(lib().ict_tracker_set_teacher(self.h_, None, 0))
            return
        poses = np.ascontiguousarray(poses, np.float32)
        assert poses.ndim == 3 and poses.shape[0] == self.T and poses.shape[2] == 8
        _check(lib().ict_tracker_set_teacher(self.h_, _p(poses), poses.shape[1]))

    def set_robust(self, flags):
        """ROBUST_FULL_STEP | ROBUST_COMPOSE | ROBUST_FLOOR: opt-in deviations from the reference (ictrack.h)."""
        _check(lib().ict_tracker_set_robust(self.h_, int(flags)))

    def set_knob(self, name, value):
        """Explicit A/B switches: "no_k2r", "seq_launches" (ictrack.h)."""
        _check(lib().ict_tracker_set_knob(self.h_, name.encode(), int(value)))

    def set_points(self, pt_off, pts, mutate_caller=False):
        """pt_off int64[T+1]; pts float64 [3*total]: per track X block, Y block, Z block."""
        pt_off = np.ascontiguousarray(pt_off, np.int64)
        assert pts.dtype == np.float64 and pts.flags.c_contiguous
        self.T = len(pt_off) - 1
        self.total = int(pt_off[-1])
        self.pt_off = pt_off
        _check(lib().ict_tracker_set_points(self.h_, self.T, _p(pt_off), _p(pts), int(mutate_caller)))

    def set_points_dev(self, T, pt_off_ptr, pts_ptr, total, max_pts, stream=0):
        self.T, self.total = T, total
        _check(lib().ict_tracker_set_points_dev(self.h_, T, C.c_void_p(pt_off_ptr), C.c_void_p(pts_ptr), total,
                                                max_pts, C.c_void_p(stream)))

    def track_batch(self, frames, ref_frame, new_frame, p_in, trace_cap=0):
        T, L = self.T, self.L
        ref_frame = np.ascontiguousarray(np.broadcast_to(ref_frame, (T,)), np.int32)
        new_frame = np.ascontiguousarray(np.broadcast_to(new_frame, (T,)), np.int32)
        p_in = np.ascontiguousarray(np.broadcast_to(p_in, (T, 6)), np.float64)
        p_out = np.zeros((T, 6), np.float64); iters = np.zeros((T, L), np.int32); npix = np.zeros(T, np.int64)
        trace = np.zeros((T, trace_cap, TRACE_FLOATS), np.float32) if trace_cap else None
        _check(lib().ict_track_batch(self.h_, frames.h_, _p(ref_frame), _p(new_frame), _p(p_in), _p(p_out), _p(iters),
                                     _p(trace), trace_cap, _p(npix)))
        return dict(p_out=p_out, iters=iters, npixres=npix, trace=trace)

    def track_batch_dev(self, frames, ref_ptr, new_ptr, p_in_ptr, p_out_ptr, iters_ptr=0, npix_ptr=0, trace_ptr=0,
                        trace_cap=0, stream=0):
        v = C.c_void_p
        _check(lib().ict_track_batch_dev(self.h_, frames.h_, v(ref_ptr), v(new_ptr), v(p_in_ptr), v(p_out_ptr),
                                         v(iters_ptr) if iters_ptr else None, v(trace_ptr) if trace_ptr else None,
                                         trace_cap, v(npix_ptr) if npix_ptr else None, v(stream)))

    def track_sequence(self, frames, first, nsteps, step, p_in):
        T, L = self.T, self.L
        p_in = np.ascontiguousarray(np.broadcast_to(p_in, (T, 6)), np.float64)
        poses = np.zeros((nsteps + 1, T, 6), np.float64)
        iters = np.zeros((max(nsteps, 1), T, L), np.int32); npix = np.zeros((max(nsteps, 1), T), np.int64)
        _check(lib().ict_track_sequence(self.h_, frames.h_, first, nsteps, step, _p(p_in), _p(poses), _p(iters),
                                        _p(npix)))
        return dict(poses=poses, iters=iters[:nsteps], npixres=npix[:nsteps])

    def reproject(self, p_in):
        """SetPose without TrackPose: the reference 2-D points at lv_l (x block, y block per track)."""
        p_in = np.ascontiguousarray(np.broadcast_to(p_in, (self.T, 6)), np.float64)
        out = np.zeros(2 * self.total, np.float32)
        _check(lib().ict_tracker_reproject(self.h_, _p(p_in), _p(out)))
        return out

    def evaluate(self, frames, ref_frame, new_frame, p_ref, p_cur=None, level=None, per_point=False):
        """One Gauss-Newton measurement per track at p_cur (default p_ref) with the template of SetPose(p_ref) at `level`
        (default lv_l), see ict_track_evaluate: dict H (T,6,6), jtr (T,6), dp (T,6), ssr (T,), nvis (T,) and, with
        per_point, pt_ssr (total,) laid out like the points (-1 where a point is not measured).  H is 4x J^T J: the
        reference's gradients are twice the derivative."""
        T = self.T
        level = self.op.lv_l if level is None else int(level)
        ref_frame = np.ascontiguousarray(np.broadcast_to(ref_frame, (T,)), np.int32)
        new_frame = np.ascontiguousarray(np.broadcast_to(new_frame, (T,)), np.int32)
        p_ref = np.ascontiguousarray(np.broadcast_to(p_ref, (T, 6)), np.float64)
        p_cur = None if p_cur is None else np.ascontiguousarray(np.broadcast_to(p_cur, (T, 6)), np.float64)
        H = np.zeros((T, 6, 6), np.float32); jtr = np.zeros((T, 6), np.float32); dp = np.zeros((T, 6), np.float32)
        ssr = np.zeros(T, np.float32); nvis = np.zeros(T, np.int32)
        pt = np.zeros(self.total, np.float32) if per_point else None
        _check(lib().ict_track_evaluate(self.h_, frames.h_, _p(ref_frame), _p(new_frame), _p(p_ref), _p(p_cur), level,
                                        _p(H), _p(jtr), _p(dp), _p(ssr), _p(nvis), _p(pt)))
        out = dict(H=H, jtr=jtr, dp=dp, ssr=ssr, nvis=nvis)
        if per_point:
            out["pt_ssr"] = pt
        return out

    def evaluate_poses(self, frames, ref_frame, new_frame, p_ref, p_cand, level=None):
        """evaluate at K candidate poses per track against the template of SetPose(p_ref) at `level` (default lv_l),
        see ict_track_evaluate_poses: p_cand (T, K, 6), broadcast like evaluate's arguments.  Returns dict H (T,6,6),
        once per track, and jtr (T,K,6), dp (T,K,6), ssr (T,K), nvis (T,K); [:, k] is evaluate(p_cur=p_cand[:, k])."""
        T = self.T
        level = self.op.lv_l if level is None else int(level)
        p_cand = np.asarray(p_cand, np.float64)
        if p_cand.ndim < 2 or p_cand.shape[-1] != 6:
            raise ValueError("p_cand must have shape (T, K, 6) or broadcast to it")
        K = p_cand.shape[-2]
        ref_frame = np.ascontiguousarray(np.broadcast_to(ref_frame, (T,)), np.int32)
        new_frame = np.ascontiguousarray(np.broadcast_to(new_frame, (T,)), np.int32)
        p_ref = np.ascontiguousarray(np.broadcast_to(p_ref, (T, 6)), np.float64)
        p_cand = np.ascontiguousarray(np.broadcast_to(p_cand, (T, K, 6)))
        H = np.zeros((T, 6, 6), np.float32); jtr = np.zeros((T, K, 6), np.float32)
        dp = np.zeros((T, K, 6), np.float32); ssr = np.zeros((T, K), np.float32); nvis = np.zeros((T, K), np.int32)
        _check(lib().ict_track_evaluate_poses(self.h_, frames.h_, _p(ref_frame), _p(new_frame), _p(p_ref), K,
                                              _p(p_cand), level, _p(H), _p(jtr), _p(dp), _p(ssr), _p(nvis)))
        return dict(H=H, jtr=jtr, dp=dp, ssr=ssr, nvis=nvis)

    def get_2dpoints(self):
        out = np.zeros(2 * self.total, np.float32)
        _check(lib().ict_tracker_get_2dpoints(self.h_, _p(out)))
        return out

    def ncc_score(self, frames, frame_b, frame_r, frame_f, nback, nfwd, pb, pr, pf):
        pb = np.ascontiguousarray(pb, np.float32); pr = np.ascontiguousarray(pr, np.float32)
        pf = np.ascontiguousarray(pf, np.float32)
        out = np.zeros(self.total, np.float32)
        _check(lib().ict_ncc_score(self.h_, frames.h_, frame_b, frame_r, frame_f, nback, nfwd, _p(pb), _p(pr), _p(pf),
                                   _p(out)))
        return out


def pose_hypotheses(fc, cc, pt2d, pt3d, sample_idx, p_init, inlthresh, maxiter=30):
    """func_ransac_fitcameras_odom.m:29-90 on the GPU: pt2d [2, n], pt3d [3, n], sample_idx [S, 4] (0-based).
    Returns dict(pose [S, 6], status [S], ninl [S], mask [S, n])."""
    fc = np.asarray(fc, np.float32); cc = np.asarray(cc, np.float32)
    pt2d = np.ascontiguousarray(pt2d, np.float64); pt3d = np.ascontiguousarray(pt3d, np.float64)
    n = pt2d.shape[1]
    assert pt2d.shape == (2, n) and pt3d.shape == (3, n)
    idx = np.ascontiguousarray(sample_idx, np.int32).reshape(-1, 4)
    S = idx.shape[0]
    p_init = np.ascontiguousarray(p_init, np.float64)
    pose = np.zeros((S, 6)); status = np.zeros(S, np.int32); ninl = np.zeros(S, np.int32); mask = np.zeros((S, n), np.uint8)
    _check(lib().ict_pose_hypotheses(fc.ctypes.data_as(_f), cc.ctypes.data_as(_f), n, _p(pt2d), _p(pt3d), S, _p(idx), _p(p_init),
                                     float(inlthresh), int(maxiter), _p(pose), _p(status), _p(ninl), _p(mask)))
    return dict(pose=pose, status=status, ninl=ninl, mask=mask)


def track_pair(op, fc, cc, wh, imgA, imgB, pts_soa, p_in, trace_cap=0):
    """Body of run_io_reprojection_test.cpp:157-224 in one call; pts_soa (float64) is centred in place if donorm."""
    fc = np.asarray(fc, np.float32); cc = np.asarray(cc, np.float32); wh = np.asarray(wh, np.int32)
    imgA = np.ascontiguousarray(imgA, np.float32); imgB = np.ascontiguousarray(imgB, np.float32)
    p_in = np.ascontiguousarray(p_in, np.float64)
    assert pts_soa.dtype == np.float64 and pts_soa.flags.c_contiguous
    L = op.lv_f - op.lv_l + 1
    p_out = np.zeros(6, np.float64); iters = np.zeros(L, np.int32)
    trace = np.zeros((trace_cap, TRACE_FLOATS), np.float32) if trace_cap else None
    _check(lib().ict_track_pair(C.byref(op), fc.ctypes.data_as(_f), cc.ctypes.data_as(_f), wh.ctypes.data_as(_i),
                                imgA.ctypes.data_as(_f), imgB.ctypes.data_as(_f), pts_soa.ctypes.data_as(_d),
                                pts_soa.size // 3, p_in.ctypes.data_as(_d), p_out.ctypes.data_as(_d), _p(iters),
                                _p(trace), trace_cap))
    return dict(p_out=p_out, iters=iters, trace=trace)
