/*
 * ictrack.h — C ABI of libictrack.so: the B200 (sm_100a) implementation of the
 * inverse-compositional Gauss-Newton pose-tracking path of catree/InvCompCamTrack.
 *
 * Convention follows the reference's only existing FFI, misc_src/triang.c as loaded by
 * misc_src/func_util_geom.py:582-604 (plain C symbols, caller-allocated contiguous buffers,
 * scalars by value, SoA layouts, results written in place).  One thing is added: every call
 * returns an int status (0 = ICT_OK) and ict_last_error() returns the message, because a GPU
 * library can fail in ways triang.c cannot.  There is NO CPU fallback behind these symbols:
 * without a CUDA device every compute entry point returns ICT_ERR_NO_DEVICE.
 *
 * Each entry point names the reference interface it replaces (file:line under the
 * reference checkout).  Names of quantities follow the reference: points (pt3d), patches,
 * steepest-descent (sd) images, Hessian, pose coefficients p = [tx ty tz wx wy wz].
 */
#ifndef ICTRACK_H
#define ICTRACK_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ICT_VERSION 100          /* 0.1.0 */
#define ICT_MAX_LEVELS 8         /* lv_f <= 7 */

enum {
  ICT_OK = 0,
  ICT_ERR_NO_DEVICE = 1,         /* no CUDA device / driver: the library never falls back to a CPU path */
  ICT_ERR_BAD_ARG = 2,
  ICT_ERR_CUDA = 3,
  ICT_ERR_NOMEM = 4,
  ICT_ERR_UNSUPPORTED = 5
};

/* Bit-compatible with CTR::optparam, utilities.h:46-61 (same field order, bool = 1 byte). */
typedef struct ict_optparam {
  int maxpttrack;                /* max points per track, multiple of 4 (run_io_reprojection_test.cpp:122-126) */
  int psz;                       /* patch size */
  int pszd2;                     /* psz/2 */
  int pszd2m3;                   /* psz + psz/2 - 1 */
  int novals;                    /* psz*psz */
  int lv_f;                      /* coarsest pyramid level (first processed) */
  int lv_l;                      /* finest pyramid level (last processed) */
  unsigned char donorm;          /* point-cloud / pose normalisation */
  unsigned char dopatchnorm;     /* patch mean subtraction */
  int maxiter;
  float normdp_ratio;
  int verbosity;
} ict_optparam;

/* Fills the derived fields the way both reference drivers do
 * (run_io_reprojection_test.cpp:112-127, run_track_nposes.cpp:47-54). */
void ict_optparam_init(ict_optparam* op, int lv_f, int lv_l, int psz, int maxiter, float normdp_ratio,
                       int donorm, int dopatchnorm, int maxpttrack, int verbosity);

int ict_version(void);
const char* ict_last_error(void);
int ict_device_count(void);                      /* 0 when no usable CUDA device */
int ict_set_device(int dev);

/* ---- a2: per-level intrinsics, CamClass::CamClass camera.cpp:14-45 -------------------------------
 * out[8*l + {0..7}] = fx fy cx cy swo sho sw sh of level l (same arithmetic: float(1/pow(2,l)) * orig). */
int ict_camera_levels(int noscales, const float fc[2], const float cc[2], const int wh[2], int padding,
                      float* out);

/* ---- a3: util_constructpyramide, utilities.cpp:14-52 ---------------------------------------------
 * Layout of one pyramid plane set: level l is a row-major (h/2^l + 2*pad) x (w/2^l + 2*pad) float plane at
 * float offset level_off[l]; returns the total number of floats of one plane set (or -1 on bad input).
 * w and h must be divisible by 2^lv_f (camera.h:12-13 states the same assumption). */
int64_t ict_pyramid_layout(int w, int h, int lv_f, int pad, int64_t* level_off, int* sw, int* sh);

/* Host image in, host planes out; the work is done on the GPU (upload, build, download). */
int ict_pyramid_build(const float* img, int w, int h, int lv_f, int pad,
                      float* out_I, float* out_dx, float* out_dy);

/* ---- device-resident frame store ------------------------------------------------------------------
 * Holds the I/dx/dy pyramids of nframes frames in HBM.  Replaces the per-frame cv::Mat arrays the drivers keep
 * (run_io_reprojection_test.cpp:143-158, run_track_nposes.cpp:157-181). */
typedef struct ict_frames ict_frames;
ict_frames* ict_frames_create(int nframes, int w, int h, int lv_f, int pad);
void ict_frames_destroy(ict_frames* fs);
/* count frames, each h*w, contiguous, from HOST memory: H2D copy + on-device pyramid build. */
int ict_frames_upload(ict_frames* fs, int first, int count, const float* imgs);
int ict_frames_upload_u8(ict_frames* fs, int first, int count, const unsigned char* imgs);   /* cv::imread(GRAYSCALE) payload */
/* Same, the images already being in device memory (float or u8); stream is a cudaStream_t (NULL = default). */
int ict_frames_build_dev(ict_frames* fs, int first, int count, const float* imgs_dev, void* stream);
int ict_frames_build_dev_u8(ict_frames* fs, int first, int count, const unsigned char* imgs_dev, void* stream);
/* Upload PRE-BUILT padded planes (what util_constructpyramide's img_ao_pyr / _dx_pyr / _dy_pyr tables point at) of
 * one frame: I/dx/dy are plane sets laid out as ict_pyramid_layout describes; dx, dy may be NULL for a frame that is
 * only ever used as the new image (SetPose takes no gradients for img_new, odometer.cpp:241). */
int ict_frames_upload_planes(ict_frames* fs, int frame, const float* I, const float* dx, const float* dy);
/* A store that owns no pixels: its entries alias frames of other stores, so that a (ref, new) pair living in two
 * stores can be handed to ict_track_batch.  Entry idx := frame src_idx of src (same w, h, lv_f, pad). */
ict_frames* ict_frames_create_view(int nframes, int w, int h, int lv_f, int pad);
int ict_frames_alias(ict_frames* view, int idx, const ict_frames* src, int src_idx);
/* Download one frame's padded planes (any of the outputs may be NULL). */
int ict_frames_download(ict_frames* fs, int frame, float* out_I, float* out_dx, float* out_dy);

/* ---- tracker: OdometerClass + PoseClass + CamClass for a BATCH of independent tracks -------------------
 * One track == one Set3Dpoints -> SetPose -> TrackPose of the reference (odometer.cpp:171-426).
 * op is copied at creation; padding of the camera == op->psz as in both drivers
 * (run_io_reprojection_test.cpp:189, run_track_nposes.cpp:185). */
typedef struct ict_tracker ict_tracker;
ict_tracker* ict_tracker_create(const ict_optparam* op, const float fc[2], const float cc[2], const int wh[2]);
void ict_tracker_destroy(ict_tracker* tr);
/* later changes of the caller's optparam (run_track_nposes.cpp:281 flips dopatchnorm mid-run).  psz and lv_f are fixed
 * at creation; lv_l, maxiter, normdp_ratio, dopatchnorm and verbosity may change between any two calls.  maxpttrack and
 * donorm shape the points that ict_tracker_set_points* stores (how many per track, and their normalisation): after a
 * change of either, the calls that read the points (tracking, reproject, get_2dpoints, ncc_score) return
 * ICT_ERR_BAD_ARG until ict_tracker_set_points* runs again.  Set both before the points, as OdometerClass does. */
int ict_tracker_set_optparam(ict_tracker* tr, const ict_optparam* op);

/* Order of the fp32 reductions (Hessian, J^T r, patch means):
 *   1 (DEFAULT) the order of Eigen 3.3's vectorised .sum() with 4-float SSE packets (eight chains per sum), which is
 *     what odometer.cpp:399-404,430-455 run when Eigen vectorises with SSE only (the model oracle/ictrack_oracle.c
 *     pins in its sum mode 0): every iteration's J^T r and delta_p, the iteration counts and the poses are
 *     bit-identical to the oracle — the mode that meets the parity gates (identical iteration counts, J^T r and pose
 *     within 1e-5).
 *   3 the same with 8-float AVX packets (sixteen chains, then predux(lo + hi)): what Eigen >= 3.3 runs when the
 *     reference is built with -mavx, as its CMakeLists.txt:4 does.  Bit-identical to the oracle in its sum mode 1.
 *     A reference binary uses one of the two; which one is found by running its driver and this library's with
 *     ICT_SUM_ORDER=1 and =3 on the same input (INTEGRATION.md).  Every tracking entry point; psz 8 and 16 run K2x8,
 *     psz 32 the general kernel (K2x / K2r have eight chains only; not measured in this order), oversized tracks the
 *     multi-CTA path.
 *   0 FAST MODE, opt-in: fixed-order parallel tree sums with the steepest-descent sums factorised per point —
 *     deterministic, 3-4x faster, equal to the reference up to fp32 summation noise (first-iteration J^T r within 4e-7
 *     of sum|sd*r|; later iterations diverge like the reference does from itself when its Eigen changes packet width:
 *     ~90 % identical iteration counts on ill-conditioned 4-point tracks, 96 % on 100-point tracks).
 *   2 tree reductions with the general kernel (any psz / dopatchnorm) even where a specialised one applies —
 *     for tests that compare the two kernels.
 * The multi-CTA path for oversized tracks honours every order, its patch means (dopatchnorm) included.  Other values:
 * ICT_ERR_BAD_ARG. */
#define ICT_SUM_ORDER_FAST 0
#define ICT_SUM_ORDER_EIGEN_SSE 1
#define ICT_SUM_ORDER_GENERAL_TREE 2
#define ICT_SUM_ORDER_EIGEN_AVX 3
int ict_tracker_set_sum_order(ict_tracker* tr, int mode);

/* ---- f3 (next row): pose hypotheses from minimal samples, func_ransac_fitcameras_odom.m:29-90 ---------------------------
 * For each of nsamples minimal samples (sample_idx[4*s + 0..3], 0-based indices into the npts 2D-3D correspondences):
 * reject degenerate samples (repeated index, three image points collinear), solve the 6-DoF pose from the four points
 * (damped Gauss-Newton on the reprojection error in fp64 from p_init, left-multiplied twists; the reference calls the
 * external ASPnP toolbox here, which is not part of its tree), reproject ALL correspondences and mark those within
 * inlthresh pixels (:48-52); a sample with fewer than four inliers is rejected (:53-57).
 *   pt2d: double[2*npts] x block, y block (pixels)      pt3d: double[3*npts] X block, Y block, Z block
 *   out_pose: double[6*nsamples] se(3) coefficients [t, w] (what run_track_nposes reads per sample)
 *   out_status: int[nsamples] 1 = usable hypothesis      out_ninl: int[nsamples] or NULL
 *   out_inlmask: uint8[nsamples*npts] or NULL
 * Host buffers; the work runs on the GPU (one thread per sample for the solve, one CTA per sample for the inliers). */
int ict_pose_hypotheses(const float fc[2], const float cc[2], int npts, const double* pt2d, const double* pt3d, int nsamples,
                        const int* sample_idx, const double p_init[6], double inlthresh, int maxiter, double* out_pose,
                        int* out_status, int* out_ninl, unsigned char* out_inlmask);

/* ---- f4 (next row): robustness modes, opt-in — NOT parity mode ----------------------------------------------------------
 * Each flag removes one documented quirk of the reference (SURVEY.md §9); results then deliberately differ from the
 * reference's.  Implemented in the fast mode for 8x8 patches (ict_tracker_set_sum_order(tr, 0), K2v8); other
 * configurations return ICT_ERR_UNSUPPORTED from the tracking calls while a flag is set.
 *   ICT_ROBUST_FULL_STEP  gradients are I(x+1) - I(x-1), twice the derivative (utilities.cpp:30-31), so every update is
 *                         half a Gauss-Newton step; this takes the full step (== halved gradients, exactly)
 *   ICT_ROBUST_COMPOSE    G <- exp(delta_p) * G instead of adding delta_p to the se(3) coefficients (pose.cpp:116-129):
 *                         the update the steepest-descent images are the derivative of
 *   ICT_ROBUST_FLOOR      patch origin floor(x) + 1 everywhere instead of ceil(x + 1e-5f) (utilities.cpp:66-69), which is
 *                         one pixel off for integer coordinates >= 256 and two for frac(x) > 1 - 1e-5
 * The fourth fix of SURVEY.md §8(f) — no stale template / steepest-descent values for points out of view — is what the
 * library does unless the knob "keep_state" asks for the reference's behaviour. */
#define ICT_ROBUST_FULL_STEP 1u
#define ICT_ROBUST_COMPOSE 2u
#define ICT_ROBUST_FLOOR 4u
int ict_tracker_set_robust(ict_tracker* tr, unsigned flags);

/* Explicit switches of a tracker (tests and A/B tools; the library reads no environment variable in its default build):
 *   "no_k2r"       1: reference-order 32x32 tracks run the producer/chain-ring kernel K2x even where K2r (resident
 *                     steepest-descent images, TMA windows) applies — same bits, for comparisons
 *   "seq_launches" 1: ict_track_sequence issues one launch per frame step even where one kernel could loop over the chain */
/*   "keep_state"   1: the reference's state between TrackPose calls (SURVEY.md §8 a4).  ResetOdometer runs only from the
 *                     constructor and Set3Dpoints (odometer.cpp:153, 173), so in the chains of
 *                     run_track_nposes.cpp:232-258 a point that has left the image keeps the template patch and
 *                     steepest-descent values of the last level — possibly of an earlier frame step — at which it was
 *                     visible, and they keep feeding the Hessian.  With this knob every ict_track_batch /
 *                     ict_track_sequence step starts from the arrays the previous call left (until the next
 *                     ict_tracker_set_points*).  Reference summation order, psz 8, up to 224 points per track (the
 *                     drivers' configuration); other configurations return ICT_ERR_UNSUPPORTED.  Default 0: every call
 *                     starts from zeroed arrays. */
int ict_tracker_set_knob(ict_tracker* tr, const char* name, int value);

/* Teacher forcing for parity tests of the fast mode (sum order 0; the reference-order kernels ignore it): poses is a host
 * array float[T * trace_cap * 8]; in the next ict_track_batch call WITH a trace of the same trace_cap, after the
 * iteration that fills trace record r of track t the pose coefficients become poses[(t*trace_cap + r)*8 + 0..5] (e.g. the
 * oracle's) instead of the kernel's own p + delta_p, and the level continues iff [.. + 6] != 0.  The trace then holds the
 * kernel's own J^T r and delta_p evaluated at the teacher's poses: identical inputs at EVERY iteration
 * (odometer.cpp:344-419).  poses == NULL clears it. */
int ict_tracker_set_teacher(ict_tracker* tr, const float* poses, int trace_cap);

/* Per-iteration trace record, ICT_TRACE_FLOATS floats:
 *   [0] level  [1] iteration  [2..7] sumsd = J^T r  [8..13] delta_p  [14] normdp  [15] #points visible in new frame
 *   [16..21] sum_k |sd_k * pdiff| — filled by the CPU oracle only (the scale fp32 summation noise is relative to;
 *            used to normalise the J^T r parity gate), 0 from the GPU
 *   [22] SM cycles of the serial solve/update section, [23] of warp 0's pixel section (production kernel only, else 0)
 * Track t owns records [t*trace_cap, (t+1)*trace_cap); unused records have level = -1. */
#define ICT_TRACE_FLOATS 24

/* Set3Dpoints for T tracks (odometer.cpp:171-239).  Track t has points pt_off[t]..pt_off[t+1]-1; its points are
 * stored as the reference expects them: X block, Y block, Z block, each of length n_t, at pts + 3*pt_off[t].
 * HOST pointers.  With donorm the reference centres the CALLER's array in place (odometer.cpp:207-212); pass
 * mutate_caller=1 to get the same side effect (pts is then written).
 * Tracks of one batch may differ in size, and a track may be empty (n_t == 0): it runs one iteration per level on no
 * pixel, its J^T r and delta_p are 0 and its pose is p_in rounded to fp32.  With donorm, a track of one point or of
 * equal points has a variance of 0 and an empty one a mean of 0/0: the reference leaves these undefined (it samples
 * the image at NaN coordinates).  Here the normalised points are NaN, and a NaN placement counts as outside the
 * image, so such a track runs one iteration per level on no pixel and returns a NaN translation and a zero rotation;
 * the CPU oracle does the same. */
int ict_tracker_set_points(ict_tracker* tr, int T, const int64_t* pt_off, double* pts, int mutate_caller);
/* Same with device pointers (pt_off_dev: int64[T+1], pts_dev: double[3*total]); nothing is written back.
 * max_pts = the largest n_t (the host needs it to size the launch). */
int ict_tracker_set_points_dev(ict_tracker* tr, int T, const int64_t* pt_off_dev, const double* pts_dev,
                               int64_t total_pts, int max_pts, void* stream);

/* SetPose + TrackPose for the T tracks set above (odometer.cpp:241-426), host buffers:
 *   ref_frame[t], new_frame[t]  indices into fs          p_in, p_out  double[T*6]
 *   iters  int[T*(lv_f-lv_l+1)] iterations run per level, coarse to fine (may be NULL)
 *   trace  float[T*trace_cap*ICT_TRACE_FLOATS] or NULL
 *   npixres int64[T] pixel-residuals evaluated per track (may be NULL). */
int ict_track_batch(ict_tracker* tr, const ict_frames* fs, const int* ref_frame, const int* new_frame,
                    const double* p_in, double* p_out, int* iters, float* trace, int trace_cap,
                    int64_t* npixres);
/* Device-pointer form; nothing crosses PCIe.  All pointers are device memory; trace_dev/iters_dev/npixres_dev
 * may be NULL. */
int ict_track_batch_dev(ict_tracker* tr, const ict_frames* fs, const int* ref_frame_dev, const int* new_frame_dev,
                        const double* p_in_dev, double* p_out_dev, int* iters_dev, float* trace_dev,
                        int trace_cap, int64_t* npixres_dev, void* stream);

/* One forward (step=+1) or backward (step=-1) chain of run_track_nposes.cpp:232-239 / :251-258 for all T tracks:
 * for k in 0..nsteps-1: SetPose(p, frame[first+k*step] as ref, frame[first+(k+1)*step] as new); TrackPose(p).
 * poses_out: double[(nsteps+1)*T*6], entry 0 = p_in. Host buffers.  The poses of the chain never leave the device
 * between steps; with 8x8 patches in the default summation order the whole chain is one kernel launch (a track's step
 * depends on its own previous step only), otherwise one launch per step: same results either way. */
int ict_track_sequence(ict_tracker* tr, const ict_frames* fs, int first, int nsteps, int step,
                       const double* p_in, double* poses_out, int* iters, int64_t* npixres);

/* SetPose WITHOUT TrackPose (run_track_nposes.cpp:217,240,259 call it only to read Get2DPoints): setpose_se3 + the
 * reference reprojection at level lv_l for all T tracks.  p_in: host double[T*6]; pt2d_out: host float[2*total],
 * laid out like ict_tracker_get_2dpoints; may be NULL (then fetch with ict_tracker_get_2dpoints). */
int ict_tracker_reproject(ict_tracker* tr, const double* p_in, float* pt2d_out);

/* Reference 2-D points of the LAST SetPose at level lv_l (OdometerClass::Get2DPoints, odometer.h:30):
 * out float[2*n_t] per track at 2*pt_off[t]: x block then y block; 0 for the points beyond maxpttrack, which the
 * reference does not project. Host buffer. */
int ict_tracker_get_2dpoints(ict_tracker* tr, float* out);

/* ---- stream-ordered host-buffer variants ------------------------------------------------------------------------
 * Same work as ict_frames_upload_u8 / ict_tracker_set_points / ict_track_batch, enqueued on the caller's
 * cudaStream_t without a final synchronisation.  Kernels and device->host copies run on that stream in call order;
 * the host->device copies of a call run on an internal copy lane of the object (its own stream; the caller's
 * stream waits for it by event, and the lane waits for the last kernel that read the copy's destination), so with
 * ONE caller stream the copies of the next chunk of a batch overlap the tracking of the current one.  Use one
 * tracker per chunk in flight and one caller stream per frame store; host buffers must be pinned (a pageable
 * source makes cudaMemcpyAsync wait for the stream) and stay valid and unmodified until the caller's stream has
 * been synchronised; outputs are valid after that.  No trace, no in-place centring of the caller's points. */
int ict_frames_upload_u8_stream(ict_frames* fs, int first, int count, const unsigned char* imgs, void* stream);
int ict_tracker_set_points_stream(ict_tracker* tr, int T, const int64_t* pt_off, const double* pts, void* stream);
int ict_track_batch_stream(ict_tracker* tr, const ict_frames* fs, const int* ref_frame, const int* new_frame,
                           const double* p_in, double* p_out, int* iters, int64_t* npixres, void* stream);

/* ---- single-pair convenience == the body of run_io_reprojection_test.cpp:157-224 -------------------
 * imgA/imgB: host h*w floats (uint8-valued as produced by imread+convertTo).  pt3d: X block, Y block, Z block
 * (npts each; written if op->donorm, like the reference).  iters/trace may be NULL. */
int ict_track_pair(const ict_optparam* op, const float fc[2], const float cc[2], const int wh[2],
                   const float* imgA, const float* imgB, double* pt3d, int npts,
                   const double p_in[6], double p_out[6], int* iters, float* trace, int trace_cap);

/* ---- a10/a11: util_getPatch / util_getPatch_grad, utilities.h:74-79, utilities.cpp:55-189 -------------------------
 * npatch bilinear psz x psz patches around mids[2*i + {0,1}] = (x, y) of level `level` of a device-resident frame:
 * the reference's placement (ceil(x + 1e-5f), origin ceil + psz/2 - padding), weights and association order; with
 * op->dopatchnorm the mean (Eigen's packet sum) is subtracted from the INTENSITY patch only (utilities.cpp:111-112,
 * 187-188).  out_I / out_dx / out_dy: host float[npatch * psz*psz], any may be NULL (util_getPatch == out_I only).
 * Centres must lie in [0, swo] x [0, sho] of the level, the range the reference samples (odometer.cpp:273-275). */
int ict_get_patches(const ict_frames* fs, int frame, int level, const ict_optparam* op, int npatch, const float* mids,
                    float* out_I, float* out_dx, float* out_dy);

/* ---- f1 (next row): NCC hypothesis scoring, run_track_nposes.cpp:271-355 ------------------------------
 * For every point of every track: mean-subtracted psz x psz patches at pt2d_back/refe/forw in frames
 * frame_b/frame_r/frame_f at level lv_l, normalised, corr = weighted max(0, dot).  pt2d_*: float[2*total] laid out
 * like ict_tracker_get_2dpoints.  out_corr: float[total]. */
int ict_ncc_score(ict_tracker* tr, const ict_frames* fs, int frame_b, int frame_r, int frame_f,
                  int nback, int nfwd, const float* pt2d_back, const float* pt2d_refe, const float* pt2d_forw,
                  float* out_corr);

/* Kernel launches issued by this library since the last reset (for bench.py's gpu_launches). */
int64_t ict_launch_count(int reset);

#ifdef __cplusplus
}
#endif
#endif /* ICTRACK_H */
