// ict_kernels.cuh — shared declarations between the kernels (ict_kernels.cu) and the C ABI (ict_capi.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/ictrack.h"

namespace ict {

// per-level intrinsics, CamClass (camera.cpp:32-43); width = (int)getsw(l) as util_getPatch receives it
struct CamLevels {
  float fx[ICT_MAX_LEVELS], fy[ICT_MAX_LEVELS], cx[ICT_MAX_LEVELS], cy[ICT_MAX_LEVELS];
  float swo[ICT_MAX_LEVELS], sho[ICT_MAX_LEVELS];
  int width[ICT_MAX_LEVELS];
};

// device pointers to the padded level planes of one frame
struct FrameDesc {
  const float* I[ICT_MAX_LEVELS];
  const float* dx[ICT_MAX_LEVELS];
  const float* dy[ICT_MAX_LEVELS];
  const void* tmap;                // device array of CUtensorMap [3 planes: I, dx, dy][ICT_MAX_LEVELS] (128 bytes each):
                                   //    2-D tiled maps of the padded level planes, box 40 x 17 floats (K2r); null when
                                   //    the geometry does not allow TMA (row pitch not a multiple of 16 bytes)
};

struct TrackParams {
  ict_optparam op;
  CamLevels cam;
  const FrameDesc* frames;
  const int* ref_frame;
  const int* new_frame;
  int fixed_ref, fixed_new;        // used when ref_frame/new_frame == nullptr (sequence chains)
  const int64_t* pt_off;           // [T+1]
  const float* pt3d;               // per track: X block, Y block, Z block (n_t each) at 3*pt_off[t]
  const double* norm;              // per track: meanshift[3], varval
  const double* p_in;              // [T*6] the SetPose pose: the template is projected at it
  const double* p_start;           // [T*6] or null (p_in): the pose TrackPose starts from (ict_track_batch_from)
  double* p_out;                   // [T*6]
  int* iters;                      // [T*L] or null
  float* trace;                    // [T*trace_cap*16] or null
  int trace_cap;
  const float* teacher;            // [T*trace_cap*8] or null (tests): teacher forcing for the fast-mode kernels — after
                                   //    iteration record r of track t the pose coefficients become teacher[(t*cap+r)*8 + 0..5]
                                   //    instead of the kernel's own p + delta_p, and the loop continues iff [6] != 0; the
                                   //    trace still records the kernel's OWN J^T r and delta_p.  Needs trace != null.
  long long* npixres;              // [T] or null
  float* pt2d_out;                 // [2*total] or null: reference 2-D points at lv_l (Get2DPoints)
  int T;                           // tracks in this launch
  int t0;                          // first track of this launch (index into the per-track arrays)
  int force_general;               // sum order 2: the multi-CTA path runs without its fused sums (tests compare the two)
  int seq_n, seq_step;             // K2v8 only: seq_n > 1 runs a whole chain in one launch — step k tracks frame
                                   //    fixed_ref + k*seq_step -> + seq_step from pose p_in + 6*T*k to p_out + 6*T*k
                                   //    (iters + T*L*k, npixres + T*k); 0/1: a single step
  float* state;                    // K2x8 with the tracker's "keep_state": per-track template state carried between calls
  int64_t state_stride;            //    (floats per track: 3*64 + 12 per point of the largest track), null: reset every call
  int state_load;                  //    0: the first call after Set3Dpoints (arrays start zeroed, odometer.cpp:173)
  unsigned robust;                 // ICT_ROBUST_* flags (ictrack.h): opt-in deviations from the reference, fast mode / psz 8 (K2v8)
  int r_pcap;                      // K2r: points per track the shared-memory layout is sized for (set by its launcher)
  int sum_mode;                    // 0: fixed-order tree reductions (fast); 1: Eigen-3.3 packet order (bit-exact
                                   //    with the oracle's default model of the reference, ~3x slower)
  int eigen_packet;                // sum_mode 1 only: float packet width of that order, 4 (SSE, eight chains per sum) or
                                   //    8 (AVX, sixteen chains); read only by code whose chain count depends on it
};

#define ICT_TRACK_SMEM_LIMIT (227 * 1024 - 8192)

// points per track a kernel's shared-memory layout holds for a track set whose largest track has max_pts points
inline int track_pcap(const ict_optparam& op, int max_pts) { return max_pts < op.maxpttrack ? max_pts : op.maxpttrack; }

int64_t launch_count(int reset);
void count_launch();               // adds one kernel launch to launch_count

// Sets kernel K's dynamic shared-memory limit and, with carveout >= 0, its preferred shared-memory carve-out (percent)
// once per device (function attributes are per device).  Templated on the kernel itself: the instances of a kernel
// template share one function-pointer type, and each needs its own attributes.
template <auto K>
cudaError_t set_kernel_attrs(int smem_limit, int carveout) {
  static bool attr_dev[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (attr_dev[dev & 63]) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(K, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_limit);
  if (e == cudaSuccess && carveout >= 0) e = cudaFuncSetAttribute(K, cudaFuncAttributePreferredSharedMemoryCarveout, carveout);
  if (e == cudaSuccess) attr_dev[dev & 63] = true;
  return e;
}

// One counted launch of the CTA-per-track kernel K, allowed up to ICT_TRACK_SMEM_LIMIT of dynamic shared memory
// (carveout as set_kernel_attrs).
template <auto K, typename... Args>
cudaError_t launch_cta_kernel(dim3 grid, int threads, size_t smem, int carveout, cudaStream_t stream,
                              const Args&... args) {
  const cudaError_t e = set_kernel_attrs<K>(ICT_TRACK_SMEM_LIMIT, carveout);
  if (e != cudaSuccess) return e;
  K<<<grid, threads, smem, stream>>>(args...);
  count_launch();
  return cudaGetLastError();
}

// ---- launches (all asynchronous on `stream`) -------------------------------------------------------------------
// K0: util_constructpyramide for `count` frames.  src is float (src_u8 == nullptr) or uint8.
cudaError_t launch_pyramid(const float* src_f32, const unsigned char* src_u8, int count, int w, int h, int lv_f,
                           int pad, float* I, float* dx, float* dy, int64_t plane_floats,
                           const int64_t* level_off, cudaStream_t stream);

// a5: Set3Dpoints for T tracks (double SoA in, float SoA + normalisation out; pts_mut gets the centred doubles)
cudaError_t launch_set_points(int T, const int64_t* pt_off, const double* pts, double* pts_mut, float* pt3d,
                              double* norm, int donorm, int maxpttrack, int max_pts, cudaStream_t stream);

// a6..a18: SetPose + TrackPose.  Every kernel below but the multi-CTA path runs one CTA per track, template +
// gradients resident in shared memory.
//   V8        k_track_v8   fast mode, psz 8 (+/- dopatchnorm); the only kernel that runs a chain of frame steps
//   V2        k_track_v2   fast mode, psz 32 without dopatchnorm
//   Fast      k_track_fast fast mode, psz 8 / 16 / 32 without dopatchnorm, where V8 and V2 do not fit
//   X8        k_track_x8   reference order, psz 8 (+/- dopatchnorm) and psz 16 without dopatchnorm
//   R         k_track_r    reference order with 4-float packets, psz 32 without dopatchnorm, needs tensor maps
//   X         k_track_x    reference order with 4-float packets, psz 32 without dopatchnorm
//   General   k_track      any psz, dopatchnorm and sum order, where its own layout fits (sum order 2: always)
//   MultiCta  launch_track_big, one track at a time
enum class TrackKernel { V8, V2, Fast, X8, R, X, General, MultiCta };
// The kernel family that runs a track set whose largest track has max_pts points.  The only place that decides it:
// a pure host function, no CUDA calls.  no_k2r and tma_ok matter only where K2r would otherwise run.
TrackKernel select_track_kernel(const ict_optparam& op, int max_pts, int sum_mode, int eigen_packet, int force_general,
                                int no_k2r, int tma_ok);
size_t track_smem_bytes(const ict_optparam& op, int max_pts, int sum_mode);
// Launches kernel k, which select_track_kernel chose for max_pts; cudaErrorInvalidConfiguration for MultiCta (the
// caller runs launch_track_big), for a chain (seq_n > 1) on any kernel but V8 and for a chain with start poses.
cudaError_t launch_track(const TrackParams& prm, TrackKernel k, int max_pts, cudaStream_t stream);

// Each kernel's own constraints: *_supported / *_smem_bytes.  The launchers assume select_track_kernel chose them.
// K2v2 (ict_kernel_v2.cu): the production kernel for psz 32 without dopatchnorm, tree sums.
size_t v2_smem_bytes(const ict_optparam& op, int max_pts);
cudaError_t launch_track_v2(const TrackParams& prm, int max_pts, cudaStream_t stream);

// K2v8 (ict_kernel_v8.cu): the K2v2 scheme for 8x8 patches (the reference's own configuration), up to 241 points per
// track, with or without dopatchnorm, tree sums; honours TrackParams.seq_n (a chain of frame steps in one launch).
bool v8_supported(const ict_optparam& op, int max_pts);
size_t v8_smem_bytes(const ict_optparam& op, int max_pts);
cudaError_t launch_track_v8(const TrackParams& prm, int max_pts, cudaStream_t stream);

// K2x (ict_kernel_x.cu): reference-order (Eigen packet) sums for psz 32 without dopatchnorm — bit-identical to the
// oracle like k_track<32,2>, with producer warps and one chain warp; 4-float packets only (eight chains).
size_t kx_smem_bytes(const ict_optparam& op, int max_pts);
cudaError_t launch_track_x(const TrackParams& prm, int max_pts, cudaStream_t stream);

// K2r (ict_kernel_r.cu): reference-order sums for psz 32 without dopatchnorm, up to 8 points per track, with the
// steepest-descent images resident in shared memory and the windows staged by 2-D TMA; needs the tensor maps (tma_ok).
bool kr_supported(const ict_optparam& op, int max_pts, int tma_ok);
size_t kr_smem_bytes(const ict_optparam& op, int max_pts);
cudaError_t launch_track_r(const TrackParams& prm, int max_pts, cudaStream_t stream);

// K2x8 (ict_kernel_x8.cu): reference-order sums for 8x8 patches (up to 222 points per track), with or without
// dopatchnorm — bit-identical to the oracle like k_track<8,2|3> (4-float packets) and k_track<8,6|7> (8-float packets).
bool kx8_supported(const ict_optparam& op, int max_pts);
size_t kx8_smem_bytes(const ict_optparam& op, int max_pts);
cudaError_t launch_track_x8(const TrackParams& prm, int max_pts, cudaStream_t stream);

// SetPose only: setpose_se3 + reprojection at lv_l into prm.pt2d_out (one CTA per track)
cudaError_t launch_reproject(const TrackParams& prm, cudaStream_t stream);

// multi-CTA path for one big track (dense alignment: psz=1, millions of points).  bigtrack_work_bytes: bytes of the
// track's work buffer; with base != null also points *out into it.
struct BigWork;
size_t bigtrack_work_bytes(const ict_optparam& op, int64_t npts, int eigen_packet, void* base = nullptr,
                           BigWork* out = nullptr);
cudaError_t launch_track_big(const TrackParams& prm, int t, int64_t npts, void* work, cudaStream_t stream);

// ict_track_evaluate (ict_evaluate.cu): one measurement per track at a chosen pose.  All pointers device memory; the
// scratch arrays are laid out by evaluate_workspace.
struct EvalPoint;
struct Lu6;
struct EvalArgs {
  ict_optparam op;
  CamLevels cam;
  const FrameDesc* frames;
  const int* ref_frame;            // [T]
  const int* new_frame;            // [T]
  const int64_t* pt_off;           // [T+1]
  const float* pt3d;               // as TrackParams.pt3d
  const double* norm;              // as TrackParams.norm
  const double* p_ref;             // [T*6] SetPose pose
  const double* p_cur;             // [T*6] measurement pose, or null: p_ref
  int T, level;
  int ref_order;                   // 1: Eigen packet order (eigen_packet 4 or 8); 0: fixed tree
  int eigen_packet;                // packet width of the reference order and of the per-point sums
  int64_t total, S;                // points, pixel slots (total * novals)
  const int64_t* chunk_off;        // [T+1] tree order: first chunk of each track
  // scratch
  float *G_ref, *G_cur;            // [T*12]
  EvalPoint* pts;                  // [total]
  float *sd, *ref, *pd;            // [6*S], [S], [S]
  float *chains, *partials;        // [T*28*2W] reference order, [chunks*28] tree order
  int* nvis;                       // [T], zeroed before the launch
  // outputs
  float *out_H, *out_jtr, *out_dp, *out_ssr, *pt_ssr;   // [T*36], [T*6], [T*6], [T], [total]
  Lu6* lu;                         // [T] each track's factorisation of H, or null (ict_track_evaluate_poses)
};
// Bytes of scratch + outputs for a's sizes (T, total, S, eigen_packet) and nchunks tree chunks; with base != null also
// points a's scratch and output pointers into it.
size_t evaluate_workspace(EvalArgs& a, int64_t nchunks, void* base);
int64_t evaluate_chunks(int64_t pixels);   // tree-order chunks of a track with that many pixel slots
cudaError_t launch_evaluate(const EvalArgs& a, int64_t nchunks, cudaStream_t stream);

// ict_track_evaluate_poses (ict_evaluate.cu): K measurements per track, one per candidate pose, against the template
// and the factorised H of SetPose(p_ref) built once per track.  The EvalArgs part carries the per-track template pass
// (p_cur null, out_jtr / out_dp / out_ssr / pt_ssr null, out_H and lu set); the candidate arrays scale with K.
struct EvalCand;
struct EvalPoses {
  int K;
  const double* p_cand;            // [T*K*6] candidate k of track t at (t*K + k)*6
  float* G_cand;                   // [T*K*12]
  EvalCand* cand;                  // [total*K] point g, candidate k at g*K + k
  float *chains, *partials;        // [T*K*7*2W] reference order, [chunks*K*7] tree order
  int* nvis;                       // [T*K], zeroed before the launch
  float *out_jtr, *out_dp, *out_ssr;   // [T*K*6], [T*K*6], [T*K]
};
size_t evaluate_poses_workspace(EvalArgs& a, EvalPoses& b, int64_t nchunks, void* base);
cudaError_t launch_evaluate_poses(const EvalArgs& a, const EvalPoses& b, int64_t nchunks, cudaStream_t stream);

// NCC hypothesis scoring, run_track_nposes.cpp:271-355
cudaError_t launch_ncc(const ict_optparam& op, const CamLevels& cam, const float* img_b, const float* img_r,
                       const float* img_f, int nback, int nfwd, const int64_t* pt_off, int T, const float* pb,
                       const float* pr, const float* pf, float* out, cudaStream_t stream);

// util_getPatch / util_getPatch_grad for npatch centres (mids: x, y pairs) on one level plane set
cudaError_t launch_get_patches(const float* I, const float* dx, const float* dy, int width, int psz, int pszd2,
                               int patchnorm, int npatch, const float* mids, float* out_I, float* out_dx, float* out_dy,
                               cudaStream_t stream);

// f3: pose hypotheses from minimal 4-point samples + inlier sets (ict_hypotheses.cu); all pointers device memory
cudaError_t launch_hypotheses(const double fc[2], const double cc[2], int npts, const double* pt2d, const double* pt3d,
                              int nsamples, const int* sample, const double p_init[6], double inlthresh, int maxiter,
                              double* pose, int* status, int* ninl, unsigned char* mask, cudaStream_t stream);

}  // namespace ict
