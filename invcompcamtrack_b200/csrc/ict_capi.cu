// ict_capi.cu — the C ABI of libictrack.so (include/ictrack.h): host-side orchestration only.
// Every compute entry point runs CUDA kernels from ict_kernels.cu; there is no CPU fallback.
#include "ict_kernels.cuh"

#include <cuda.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>

using namespace ict;

// ---------------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CU(expr)                                                                                       \
  do {                                                                                                 \
    cudaError_t _e = (expr);                                                                           \
    if (_e != cudaSuccess)                                                                             \
      return fail(ICT_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));                   \
  } while (0)

static int require_device() {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    cudaGetLastError();
    return fail(ICT_ERR_NO_DEVICE, "no CUDA device: libictrack has no CPU fallback");
  }
  return ICT_OK;
}

// grow-only device buffer
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T> T* as() const { return (T*)p; }
};

// Internal copy lane of the *_stream entry points.  Host->device copies of a call run on the object's own stream and
// the caller's stream waits for them by event, so the copy of call k+1 overlaps whatever the caller's stream is
// still executing for call k, while every KERNEL stays on the caller's one stream in call order.  (Kernels of two
// calls on two caller streams do overlap, but badly: the small pyramid CTAs of the next chunk take the slots that
// tracking CTAs free one by one and run at a fraction of their normal occupancy — measured +0.7 ms per 6.2 ms chunk,
// profiles/tools/e2e_timeline.py.)  `consumed` is recorded on the caller's stream after the last kernel that reads the
// copy's destination; the lane waits for it before overwriting the destination in a later call.
struct CopyLane {
  cudaStream_t s = nullptr;
  cudaEvent_t copied = nullptr, consumed = nullptr;
  bool have_consumed = false;
  cudaError_t begin() {                     // call before the copies of one API call
    cudaError_t e = cudaSuccess;
    if (!s) {
      e = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
      if (e == cudaSuccess) e = cudaEventCreateWithFlags(&copied, cudaEventDisableTiming);
      if (e == cudaSuccess) e = cudaEventCreateWithFlags(&consumed, cudaEventDisableTiming);
      if (e != cudaSuccess) return e;
    }
    if (have_consumed) e = cudaStreamWaitEvent(s, consumed, 0);
    return e;
  }
  cudaError_t publish(cudaStream_t user) {  // after the copies: the caller's stream sees them
    cudaError_t e = cudaEventRecord(copied, s);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(user, copied, 0);
    return e;
  }
  cudaError_t done(cudaStream_t user) {     // after the last kernel that reads the copied data
    if (!s) return cudaSuccess;             // the lane never copied anything (points set by a blocking / device call)
    cudaError_t e = cudaEventRecord(consumed, user);
    have_consumed = e == cudaSuccess;
    return e;
  }
  void release() {
    if (s) {
      cudaStreamSynchronize(s);
      cudaEventDestroy(copied);
      cudaEventDestroy(consumed);
      cudaStreamDestroy(s);
      s = nullptr;
    }
  }
};

extern "C" {

// ---------------------------------------------------------------------------------------------------
void ict_optparam_init(ict_optparam* op, int lv_f, int lv_l, int psz, int maxiter, float normdp_ratio, int donorm,
                       int dopatchnorm, int maxpttrack, int verbosity) {
  memset(op, 0, sizeof(*op));
  op->lv_f = lv_f;
  op->lv_l = lv_l;
  op->psz = psz;
  op->pszd2 = psz / 2;                 // run_io_reprojection_test.cpp:115
  op->pszd2m3 = psz + op->pszd2 - 1;   // :116
  op->novals = psz * psz;              // :117
  op->maxiter = maxiter;
  op->normdp_ratio = normdp_ratio;
  op->donorm = donorm ? 1 : 0;
  op->dopatchnorm = dopatchnorm ? 1 : 0;
  const int r = maxpttrack % 4;        // SSEMULTIPL padding, :123-126
  op->maxpttrack = r > 0 ? maxpttrack + (4 - r) : maxpttrack;
  op->verbosity = verbosity;
}

int ict_version(void) { return ICT_VERSION; }
const char* ict_last_error(void) { return g_err.c_str(); }

int ict_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int ict_set_device(int dev) {
  if (require_device()) return ICT_ERR_NO_DEVICE;
  CU(cudaSetDevice(dev));
  return ICT_OK;
}

int64_t ict_launch_count(int reset) { return launch_count(reset); }

// ---- camera (camera.cpp:32-43) ------------------------------------------------------------------------
int ict_camera_levels(int noscales, const float fc[2], const float cc[2], const int wh[2], int padding,
                      float* out) {
  if (noscales < 1 || noscales > ICT_MAX_LEVELS) return fail(ICT_ERR_BAD_ARG, "noscales out of range");
  for (int i = 0; i < noscales; ++i) {
    const float sc_fct = (float)(1 / pow(2, i));
    float* o = out + 8 * i;
    o[0] = sc_fct * fc[0];
    o[1] = sc_fct * fc[1];
    o[2] = sc_fct * cc[0];
    o[3] = sc_fct * cc[1];
    o[4] = sc_fct * (float)wh[0];
    o[5] = sc_fct * (float)wh[1];
    o[6] = o[4] + 2 * padding;
    o[7] = o[5] + 2 * padding;
  }
  return ICT_OK;
}

static void fill_cam(CamLevels& cam, int noscales, const float fc[2], const float cc[2], const int wh[2],
                     int padding) {
  float lv[8 * ICT_MAX_LEVELS];
  ict_camera_levels(noscales, fc, cc, wh, padding, lv);
  memset(&cam, 0, sizeof(cam));
  for (int l = 0; l < noscales; ++l) {
    cam.fx[l] = lv[8 * l + 0];
    cam.fy[l] = lv[8 * l + 1];
    cam.cx[l] = lv[8 * l + 2];
    cam.cy[l] = lv[8 * l + 3];
    cam.swo[l] = lv[8 * l + 4];
    cam.sho[l] = lv[8 * l + 5];
    cam.width[l] = (int)lv[8 * l + 6];   // float getsw() received as `const int width`, odometer.cpp:286
  }
}

// ---- pyramid ------------------------------------------------------------------------------------------
int64_t ict_pyramid_layout(int w, int h, int lv_f, int pad, int64_t* level_off, int* sw, int* sh) {
  if (w <= 0 || h <= 0 || lv_f < 0 || lv_f >= ICT_MAX_LEVELS || pad < 0) return -1;
  if ((w % (1 << lv_f)) || (h % (1 << lv_f))) return -1;   // camera.h:12-13: sizes divisible by 2 per level
  int64_t tot = 0;
  for (int l = 0; l <= lv_f; ++l) {
    const int a = (w >> l) + 2 * pad, b = (h >> l) + 2 * pad;
    if (level_off) level_off[l] = tot;
    if (sw) sw[l] = a;
    if (sh) sh[l] = b;
    tot += (int64_t)a * b;
  }
  return tot;
}

struct ict_frames {
  int nframes, w, h, lv_f, pad;
  int64_t plane_floats;
  int64_t level_off[ICT_MAX_LEVELS];
  int sw[ICT_MAX_LEVELS], sh[ICT_MAX_LEVELS];
  float *I, *dx, *dy;
  FrameDesc* desc;
  void* tmaps;        // device: CUtensorMap [nframes][3 planes][ICT_MAX_LEVELS], or null (geometry not TMA-able)
  bool tma_ok;        // every entry of desc carries tensor maps (a view: every frame aliased so far does)
  DevBuf stage;
  CopyLane lane;
  bool view;
};

// ---- tensor maps of the padded level planes (K2r stages its windows with cp.async.bulk.tensor.2d) --------------------
// One 2-D tiled map per frame, plane (I, dx, dy) and level: dimensions (sw, sh) floats, row pitch sw * 4 bytes, box
// 40 x 17 floats = one half-patch window of a 32x32 patch (row above + 16 rows; column to the left + 32, starting at a
// multiple of four columns because the innermost TMA coordinate has to be 16-byte aligned), no swizzle, no interleave.  TMA wants a 16-byte aligned base and a row pitch that
// is a multiple of 16 bytes: with pad == 32 that holds whenever (w >> l) is a multiple of 4 on every level.
// cuTensorMapEncodeTiled is reached through the runtime's driver entry point query: libictrack.so does not link
// libcuda.
typedef CUresult (*ict_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static ict_encode_tiled_fn encode_tiled_fn() {
  static ict_encode_tiled_fn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (ict_encode_tiled_fn)p;
    else
      cudaGetLastError();
  }
  return fn;
}

#define ICT_TMA_BOX_W 40
#define ICT_TMA_BOX_H 17

static bool frames_make_tmaps(ict_frames* fs) {
  fs->tmaps = nullptr;
  fs->tma_ok = false;
  if (fs->pad != 32) return false;               // the box is the half-patch window of a 32x32 patch
  ict_encode_tiled_fn enc = encode_tiled_fn();
  if (!enc) return false;
  for (int l = 0; l <= fs->lv_f; ++l)
    if ((fs->sw[l] % 4) || (fs->level_off[l] % 4) || fs->sw[l] < ICT_TMA_BOX_W || fs->sh[l] < ICT_TMA_BOX_H) return false;
  if (fs->plane_floats % 4) return false;
  const size_t per_frame = 3 * ICT_MAX_LEVELS;
  std::vector<CUtensorMap> maps(per_frame * fs->nframes);
  memset(maps.data(), 0, sizeof(CUtensorMap) * maps.size());
  float* planes[3] = {fs->I, fs->dx, fs->dy};
  for (int f = 0; f < fs->nframes; ++f)
    for (int q = 0; q < 3; ++q)
      for (int l = 0; l <= fs->lv_f; ++l) {
        void* base = planes[q] + (size_t)f * fs->plane_floats + fs->level_off[l];
        const cuuint64_t dims[2] = {(cuuint64_t)fs->sw[l], (cuuint64_t)fs->sh[l]};
        const cuuint64_t strides[1] = {(cuuint64_t)fs->sw[l] * sizeof(float)};
        const cuuint32_t box[2] = {ICT_TMA_BOX_W, ICT_TMA_BOX_H};
        const cuuint32_t estr[2] = {1, 1};
        if (enc(&maps[(f * 3 + q) * ICT_MAX_LEVELS + l], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box, estr,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
          return false;
      }
  if (cudaMalloc(&fs->tmaps, sizeof(CUtensorMap) * maps.size()) != cudaSuccess) {
    cudaGetLastError();
    fs->tmaps = nullptr;
    return false;
  }
  if (cudaMemcpy(fs->tmaps, maps.data(), sizeof(CUtensorMap) * maps.size(), cudaMemcpyHostToDevice) != cudaSuccess) {
    cudaFree(fs->tmaps);
    fs->tmaps = nullptr;
    return false;
  }
  fs->tma_ok = true;
  return true;
}

ict_frames* ict_frames_create(int nframes, int w, int h, int lv_f, int pad) {
  if (require_device()) return nullptr;
  ict_frames* fs = new ict_frames();
  fs->nframes = nframes; fs->w = w; fs->h = h; fs->lv_f = lv_f; fs->pad = pad;
  fs->I = fs->dx = fs->dy = nullptr;
  fs->desc = nullptr;
  fs->tmaps = nullptr;
  fs->tma_ok = false;
  fs->view = false;
  fs->plane_floats = ict_pyramid_layout(w, h, lv_f, pad, fs->level_off, fs->sw, fs->sh);
  if (fs->plane_floats < 0 || nframes <= 0) {
    fail(ICT_ERR_BAD_ARG, "ict_frames_create: w,h must be divisible by 2^lv_f, nframes > 0");
    delete fs;
    return nullptr;
  }
  const size_t bytes = sizeof(float) * (size_t)fs->plane_floats * nframes;
  if (cudaMalloc(&fs->I, bytes) != cudaSuccess || cudaMalloc(&fs->dx, bytes) != cudaSuccess ||
      cudaMalloc(&fs->dy, bytes) != cudaSuccess || cudaMalloc(&fs->desc, sizeof(FrameDesc) * nframes) != cudaSuccess) {
    fail(ICT_ERR_NOMEM, "ict_frames_create: cudaMalloc failed");
    cudaGetLastError();
    ict_frames_destroy(fs);
    return nullptr;
  }
  frames_make_tmaps(fs);       // optional: without them the reference-order path of psz 32 runs K2x instead of K2r
  std::vector<FrameDesc> d(nframes);
  for (int f = 0; f < nframes; ++f) {
    memset(&d[f], 0, sizeof(FrameDesc));
    d[f].tmap = fs->tmaps ? (const char*)fs->tmaps + sizeof(CUtensorMap) * 3 * ICT_MAX_LEVELS * (size_t)f : nullptr;
    for (int l = 0; l <= lv_f; ++l) {
      d[f].I[l] = fs->I + (size_t)f * fs->plane_floats + fs->level_off[l];
      d[f].dx[l] = fs->dx + (size_t)f * fs->plane_floats + fs->level_off[l];
      d[f].dy[l] = fs->dy + (size_t)f * fs->plane_floats + fs->level_off[l];
    }
  }
  if (cudaMemcpy(fs->desc, d.data(), sizeof(FrameDesc) * nframes, cudaMemcpyHostToDevice) != cudaSuccess) {
    fail(ICT_ERR_CUDA, "ict_frames_create: descriptor upload failed");
    ict_frames_destroy(fs);
    return nullptr;
  }
  return fs;
}

void ict_frames_destroy(ict_frames* fs) {
  if (!fs) return;
  if (fs->I) cudaFree(fs->I);
  if (fs->dx) cudaFree(fs->dx);
  if (fs->dy) cudaFree(fs->dy);
  if (fs->desc) cudaFree(fs->desc);
  if (fs->tmaps) cudaFree(fs->tmaps);
  fs->stage.release();
  fs->lane.release();
  delete fs;
}

ict_frames* ict_frames_create_view(int nframes, int w, int h, int lv_f, int pad) {
  if (require_device()) return nullptr;
  ict_frames* fs = new ict_frames();
  fs->nframes = nframes; fs->w = w; fs->h = h; fs->lv_f = lv_f; fs->pad = pad;
  fs->I = fs->dx = fs->dy = nullptr;
  fs->desc = nullptr;
  fs->tmaps = nullptr;
  fs->tma_ok = true;           // until a frame without tensor maps is aliased
  fs->view = true;
  fs->plane_floats = ict_pyramid_layout(w, h, lv_f, pad, fs->level_off, fs->sw, fs->sh);
  if (fs->plane_floats < 0 || nframes <= 0 || cudaMalloc(&fs->desc, sizeof(FrameDesc) * nframes) != cudaSuccess) {
    fail(ICT_ERR_BAD_ARG, "ict_frames_create_view: bad geometry or allocation failure");
    cudaGetLastError();
    delete fs;
    return nullptr;
  }
  cudaMemset(fs->desc, 0, sizeof(FrameDesc) * nframes);
  return fs;
}

int ict_frames_alias(ict_frames* view, int idx, const ict_frames* src, int src_idx) {
  if (!view || !src || !view->view) return fail(ICT_ERR_BAD_ARG, "ict_frames_alias: first argument must be a view store");
  if (idx < 0 || idx >= view->nframes || src_idx < 0 || src_idx >= src->nframes)
    return fail(ICT_ERR_BAD_ARG, "ict_frames_alias: index out of range");
  if (view->w != src->w || view->h != src->h || view->lv_f != src->lv_f || view->pad != src->pad)
    return fail(ICT_ERR_BAD_ARG, "ict_frames_alias: geometry mismatch");
  CU(cudaMemcpyAsync(view->desc + idx, src->desc + src_idx, sizeof(FrameDesc), cudaMemcpyDeviceToDevice, 0));
  view->tma_ok = view->tma_ok && src->tma_ok;
  return ICT_OK;
}

static int frames_range_ok(const ict_frames* fs, int first, int count) {
  if (!fs) return fail(ICT_ERR_BAD_ARG, "null frame store");
  if (first < 0 || count < 0 || first + count > fs->nframes) return fail(ICT_ERR_BAD_ARG, "frame range out of bounds");
  return ICT_OK;
}

static int frames_build(ict_frames* fs, int first, int count, const float* f32, const unsigned char* u8,
                        cudaStream_t st) {
  if (fs->view) return fail(ICT_ERR_BAD_ARG, "a view store owns no pixels: build into the store it aliases");
  CU(launch_pyramid(f32, u8, count, fs->w, fs->h, fs->lv_f, fs->pad, fs->I + (size_t)first * fs->plane_floats,
                    fs->dx + (size_t)first * fs->plane_floats, fs->dy + (size_t)first * fs->plane_floats,
                    fs->plane_floats, fs->level_off, st));
  return ICT_OK;
}

int ict_frames_build_dev(ict_frames* fs, int first, int count, const float* imgs_dev, void* stream) {
  if (frames_range_ok(fs, first, count)) return ICT_ERR_BAD_ARG;
  return frames_build(fs, first, count, imgs_dev, nullptr, (cudaStream_t)stream);
}
int ict_frames_build_dev_u8(ict_frames* fs, int first, int count, const unsigned char* imgs_dev, void* stream) {
  if (frames_range_ok(fs, first, count)) return ICT_ERR_BAD_ARG;
  return frames_build(fs, first, count, nullptr, imgs_dev, (cudaStream_t)stream);
}

int ict_frames_upload(ict_frames* fs, int first, int count, const float* imgs) {
  if (frames_range_ok(fs, first, count)) return ICT_ERR_BAD_ARG;
  const size_t bytes = sizeof(float) * (size_t)fs->w * fs->h * count;
  CU(fs->stage.reserve(bytes));
  CU(cudaMemcpyAsync(fs->stage.p, imgs, bytes, cudaMemcpyHostToDevice, 0));
  return frames_build(fs, first, count, fs->stage.as<float>(), nullptr, 0);
}
int ict_frames_upload_u8(ict_frames* fs, int first, int count, const unsigned char* imgs) {
  if (frames_range_ok(fs, first, count)) return ICT_ERR_BAD_ARG;
  const size_t bytes = (size_t)fs->w * fs->h * count;
  CU(fs->stage.reserve(bytes));
  CU(cudaMemcpyAsync(fs->stage.p, imgs, bytes, cudaMemcpyHostToDevice, 0));
  return frames_build(fs, first, count, nullptr, fs->stage.as<unsigned char>(), 0);
}

int ict_frames_upload_planes(ict_frames* fs, int frame, const float* I, const float* dx, const float* dy) {
  if (frames_range_ok(fs, frame, 1)) return ICT_ERR_BAD_ARG;
  if (fs->view || !I) return fail(ICT_ERR_BAD_ARG, "ict_frames_upload_planes: needs an owning store and an intensity plane set");
  const size_t bytes = sizeof(float) * (size_t)fs->plane_floats, o = (size_t)frame * fs->plane_floats;
  CU(cudaMemcpyAsync(fs->I + o, I, bytes, cudaMemcpyHostToDevice, 0));
  if (dx) CU(cudaMemcpyAsync(fs->dx + o, dx, bytes, cudaMemcpyHostToDevice, 0));
  if (dy) CU(cudaMemcpyAsync(fs->dy + o, dy, bytes, cudaMemcpyHostToDevice, 0));
  CU(cudaStreamSynchronize(0));
  return ICT_OK;
}

int ict_frames_upload_u8_stream(ict_frames* fs, int first, int count, const unsigned char* imgs, void* stream) {
  if (frames_range_ok(fs, first, count)) return ICT_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t per = (size_t)fs->w * fs->h;
  // one staging area for the whole store, each frame at its own offset: chunks in flight never share bytes
  if (fs->stage.cap < per * fs->nframes) {
    CU(cudaDeviceSynchronize());
    CU(fs->stage.reserve(per * fs->nframes));
  }
  unsigned char* dst = fs->stage.as<unsigned char>() + per * first;
  CU(fs->lane.begin());
  CU(cudaMemcpyAsync(dst, imgs, per * count, cudaMemcpyHostToDevice, fs->lane.s));
  CU(fs->lane.publish(st));
  const int rc = frames_build(fs, first, count, nullptr, dst, st);
  if (rc) return rc;
  CU(fs->lane.done(st));
  return ICT_OK;
}

int ict_frames_download(ict_frames* fs, int frame, float* out_I, float* out_dx, float* out_dy) {
  if (frames_range_ok(fs, frame, 1)) return ICT_ERR_BAD_ARG;
  if (fs->view) return fail(ICT_ERR_BAD_ARG, "ict_frames_download: a view store owns no pixels");
  const size_t bytes = sizeof(float) * (size_t)fs->plane_floats, o = (size_t)frame * fs->plane_floats;
  if (out_I) CU(cudaMemcpy(out_I, fs->I + o, bytes, cudaMemcpyDeviceToHost));
  if (out_dx) CU(cudaMemcpy(out_dx, fs->dx + o, bytes, cudaMemcpyDeviceToHost));
  if (out_dy) CU(cudaMemcpy(out_dy, fs->dy + o, bytes, cudaMemcpyDeviceToHost));
  return ICT_OK;
}

int ict_pyramid_build(const float* img, int w, int h, int lv_f, int pad, float* out_I, float* out_dx,
                      float* out_dy) {
  if (require_device()) return ICT_ERR_NO_DEVICE;
  ict_frames* fs = ict_frames_create(1, w, h, lv_f, pad);
  if (!fs) return ICT_ERR_BAD_ARG;
  int rc = ict_frames_upload(fs, 0, 1, img);
  if (rc == ICT_OK) rc = ict_frames_download(fs, 0, out_I, out_dx, out_dy);
  ict_frames_destroy(fs);
  return rc;
}

// ---- tracker ------------------------------------------------------------------------------------------
struct ict_tracker {
  ict_optparam op;
  CamLevels cam;
  float fc[2], cc[2];
  int wh[2];
  int T = 0;
  int64_t total = 0;
  int max_pts = 0;
  int pts_maxpttrack = 0, pts_donorm = 0;   // the optparam fields ict_tracker_set_points* stored the points with
  std::vector<int64_t> h_off;
  bool have_2d = false;
  int sum_mode = 1;            // the reference's summation order is the default (ictrack.h, ict_tracker_set_sum_order)
  int eigen_packet = 4;        // float packet width of that order: 4 (SSE, the default) or 8 (AVX, sum order 3)
  int force_general = 0;
  int knob_no_k2r = 0, knob_seq_launches = 0;   // ict_tracker_set_knob
  unsigned robust = 0;         // ict_tracker_set_robust
  int keep_state = 0;          // knob "keep_state": template arrays persist between TrackPose calls until the next Set3Dpoints
  bool state_valid = false;
  int seq_n = 0, seq_step = 0;   // set by ict_track_sequence around one run_tracks call (chain in one launch)
  const int *big_rf = nullptr, *big_nf = nullptr;   // set by ict_track_batch around run_tracks: per-track frames (host) of the multi-CTA path
  DevBuf pt_off, pts, pt3d, norm, p_in, p_out, iters, npix, trace, pt2d, rf, nf, big, teacher, state;
  int teacher_cap = 0;           // ict_tracker_set_teacher: records per track of the staged teacher poses (0: none)
  // several multi-CTA tracks in one call run on up to ICT_BIG_LANES streams side by side (each track is a chain of a few
  // hundred small launches: their latencies overlap); every lane has its own work buffer
  static const int ICT_BIG_LANES = 4;
  cudaStream_t big_st[ICT_BIG_LANES] = {};
  cudaEvent_t big_ev[ICT_BIG_LANES + 1] = {};
  DevBuf big_lane[ICT_BIG_LANES];
  CopyLane lane;      // points (ict_tracker_set_points_stream)
  CopyLane lane_in;   // per-call inputs of ict_track_batch_stream: frame indices, initial poses
};

static bool optparam_ok(const ict_optparam* op) {
  return op && op->psz >= 1 && op->lv_f >= op->lv_l && op->lv_l >= 0 && op->lv_f < ICT_MAX_LEVELS && op->maxpttrack >= 1 &&
         op->maxiter >= 0;
}

ict_tracker* ict_tracker_create(const ict_optparam* op, const float fc[2], const float cc[2], const int wh[2]) {
  if (require_device()) return nullptr;
  if (!optparam_ok(op) || !fc || !cc || !wh) {
    fail(ICT_ERR_BAD_ARG, "ict_tracker_create: bad optparam");
    return nullptr;
  }
  ict_tracker* tr = new ict_tracker();
  tr->op = *op;
  memcpy(tr->fc, fc, sizeof(tr->fc));
  memcpy(tr->cc, cc, sizeof(tr->cc));
  memcpy(tr->wh, wh, sizeof(tr->wh));
  fill_cam(tr->cam, op->lv_f + 1, fc, cc, wh, op->psz);   // padding = psz, run_io_reprojection_test.cpp:189
  return tr;
}

void ict_tracker_destroy(ict_tracker* tr) {
  if (!tr) return;
  DevBuf* b[] = {&tr->pt_off, &tr->pts, &tr->pt3d, &tr->norm, &tr->p_in, &tr->p_out, &tr->iters,
                 &tr->npix, &tr->trace, &tr->pt2d, &tr->rf, &tr->nf, &tr->big, &tr->teacher, &tr->state};
  for (DevBuf* x : b) x->release();
  for (int k = 0; k < ict_tracker::ICT_BIG_LANES; ++k) {
    tr->big_lane[k].release();
    if (tr->big_st[k]) cudaStreamDestroy(tr->big_st[k]);
  }
  for (int k = 0; k <= ict_tracker::ICT_BIG_LANES; ++k)
    if (tr->big_ev[k]) cudaEventDestroy(tr->big_ev[k]);
  tr->lane.release();
  tr->lane_in.release();
  delete tr;
}

int ict_tracker_set_optparam(ict_tracker* tr, const ict_optparam* op) {
  if (!tr || !op) return fail(ICT_ERR_BAD_ARG, "null argument");
  if (op->psz != tr->op.psz || op->lv_f != tr->op.lv_f)
    return fail(ICT_ERR_BAD_ARG, "psz and lv_f are fixed at creation (they size the camera and the pyramids)");
  if (!optparam_ok(op)) return fail(ICT_ERR_BAD_ARG, "ict_tracker_set_optparam: bad optparam (lv_l, maxpttrack or maxiter out of range)");
  tr->op = *op;
  tr->op.pszd2 = op->psz / 2;                      // the derived fields follow psz (run_io_reprojection_test.cpp:115-117)
  tr->op.pszd2m3 = op->psz + op->psz / 2 - 1;
  tr->op.novals = op->psz * op->psz;
  return ICT_OK;
}

int ict_tracker_set_teacher(ict_tracker* tr, const float* poses, int trace_cap) {
  if (!tr) return fail(ICT_ERR_BAD_ARG, "null argument");
  if (!poses || trace_cap <= 0) {
    tr->teacher_cap = 0;
    return ICT_OK;
  }
  if (tr->T <= 0) return fail(ICT_ERR_BAD_ARG, "no points set");
  const size_t bytes = sizeof(float) * 8 * (size_t)tr->T * trace_cap;
  CU(tr->teacher.reserve(bytes));
  CU(cudaMemcpy(tr->teacher.p, poses, bytes, cudaMemcpyHostToDevice));
  tr->teacher_cap = trace_cap;
  return ICT_OK;
}

int ict_tracker_set_robust(ict_tracker* tr, unsigned flags) {
  if (!tr || (flags & ~(ICT_ROBUST_FULL_STEP | ICT_ROBUST_COMPOSE | ICT_ROBUST_FLOOR)))
    return fail(ICT_ERR_BAD_ARG, "ict_tracker_set_robust: unknown flag");
  tr->robust = flags;
  return ICT_OK;
}

int ict_tracker_set_knob(ict_tracker* tr, const char* name, int value) {
  if (!tr || !name) return fail(ICT_ERR_BAD_ARG, "null argument");
  if (!strcmp(name, "no_k2r")) tr->knob_no_k2r = value ? 1 : 0;
  else if (!strcmp(name, "seq_launches")) tr->knob_seq_launches = value ? 1 : 0;
  else if (!strcmp(name, "keep_state")) { tr->keep_state = value ? 1 : 0; tr->state_valid = false; }
  else return fail(ICT_ERR_BAD_ARG, std::string("unknown knob: ") + name);
  return ICT_OK;
}

int ict_tracker_set_sum_order(ict_tracker* tr, int mode) {
  if (!tr || mode < 0 || mode > 3)
    return fail(ICT_ERR_BAD_ARG, "sum order must be 1 (reference order, 4-float packets, default), 3 (reference order, "
                                 "8-float packets), 0 (fast tree order) or 2");
  tr->sum_mode = (mode == 1 || mode == 3) ? 1 : 0;
  tr->eigen_packet = mode == 3 ? 8 : 4;
  tr->force_general = mode == 2 ? 1 : 0;
  return ICT_OK;
}

static int tracker_reserve(ict_tracker* tr, int T, int64_t total, cudaStream_t st) {
  CU(tr->pt_off.reserve(sizeof(int64_t) * (size_t)(T + 1)));
  CU(tr->pt3d.reserve(sizeof(float) * 3 * (size_t)(total ? total : 1)));
  CU(tr->norm.reserve(sizeof(double) * 4 * (size_t)T));
  CU(tr->pt2d.reserve(sizeof(float) * 2 * (size_t)(total ? total : 1)));
  // no kernel writes the 2-D points of a track's points beyond maxpttrack: they read 0, not a reused buffer's contents
  CU(cudaMemsetAsync(tr->pt2d.p, 0, sizeof(float) * 2 * (size_t)total, st));
  return ICT_OK;
}

int ict_tracker_set_points(ict_tracker* tr, int T, const int64_t* pt_off, double* pts, int mutate_caller) {
  if (!tr || T <= 0 || !pt_off || !pts) return fail(ICT_ERR_BAD_ARG, "ict_tracker_set_points: bad argument");
  const int64_t total = pt_off[T];
  int max_pts = 0;
  for (int t = 0; t < T; ++t) {
    const int64_t n = pt_off[t + 1] - pt_off[t];
    if (n < 0 || n > 0x7fffffff) return fail(ICT_ERR_BAD_ARG, "pt_off must be non-decreasing");
    if (n > max_pts) max_pts = (int)n;
  }
  if (tracker_reserve(tr, T, total, 0)) return ICT_ERR_CUDA;
  CU(tr->pts.reserve(sizeof(double) * 3 * (size_t)(total ? total : 1)));
  CU(cudaMemcpyAsync(tr->pt_off.p, pt_off, sizeof(int64_t) * (size_t)(T + 1), cudaMemcpyHostToDevice, 0));
  CU(cudaMemcpyAsync(tr->pts.p, pts, sizeof(double) * 3 * (size_t)total, cudaMemcpyHostToDevice, 0));
  const bool mut = mutate_caller && tr->op.donorm;
  CU(launch_set_points(T, tr->pt_off.as<int64_t>(), tr->pts.as<double>(), mut ? tr->pts.as<double>() : nullptr,
                       tr->pt3d.as<float>(), tr->norm.as<double>(), tr->op.donorm, tr->op.maxpttrack, max_pts, 0));
  if (mut) CU(cudaMemcpy(pts, tr->pts.p, sizeof(double) * 3 * (size_t)total, cudaMemcpyDeviceToHost));
  tr->T = T;
  tr->total = total;
  tr->max_pts = max_pts;
  tr->pts_maxpttrack = tr->op.maxpttrack;
  tr->pts_donorm = tr->op.donorm;
  tr->h_off.assign(pt_off, pt_off + T + 1);
  tr->have_2d = false;
  tr->state_valid = false;     // Set3Dpoints resets the odometer (odometer.cpp:173)
  return ICT_OK;
}

int ict_tracker_set_points_stream(ict_tracker* tr, int T, const int64_t* pt_off, const double* pts, void* stream) {
  if (!tr || T <= 0 || !pt_off || !pts) return fail(ICT_ERR_BAD_ARG, "ict_tracker_set_points_stream: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t total = pt_off[T];
  int max_pts = 0;
  for (int t = 0; t < T; ++t) {
    const int64_t n = pt_off[t + 1] - pt_off[t];
    if (n < 0 || n > 0x7fffffff) return fail(ICT_ERR_BAD_ARG, "pt_off must be non-decreasing");
    if (n > max_pts) max_pts = (int)n;
  }
  if (tracker_reserve(tr, T, total, st)) return ICT_ERR_CUDA;
  CU(tr->pts.reserve(sizeof(double) * 3 * (size_t)(total ? total : 1)));
  CU(tr->lane.begin());
  CU(cudaMemcpyAsync(tr->pt_off.p, pt_off, sizeof(int64_t) * (size_t)(T + 1), cudaMemcpyHostToDevice, tr->lane.s));
  CU(cudaMemcpyAsync(tr->pts.p, pts, sizeof(double) * 3 * (size_t)total, cudaMemcpyHostToDevice, tr->lane.s));
  CU(tr->lane.publish(st));
  CU(launch_set_points(T, tr->pt_off.as<int64_t>(), tr->pts.as<double>(), nullptr, tr->pt3d.as<float>(),
                       tr->norm.as<double>(), tr->op.donorm, tr->op.maxpttrack, max_pts, st));
  CU(tr->lane.done(st));   // pt_off stays in use by later tracking calls: ict_track_batch_stream records again
  tr->T = T;
  tr->total = total;
  tr->max_pts = max_pts;
  tr->pts_maxpttrack = tr->op.maxpttrack;
  tr->pts_donorm = tr->op.donorm;
  tr->h_off.assign(pt_off, pt_off + T + 1);
  tr->have_2d = false;
  tr->state_valid = false;     // Set3Dpoints resets the odometer (odometer.cpp:173)
  return ICT_OK;
}

int ict_tracker_set_points_dev(ict_tracker* tr, int T, const int64_t* pt_off_dev, const double* pts_dev,
                               int64_t total_pts, int max_pts, void* stream) {
  if (!tr || T <= 0 || !pt_off_dev || !pts_dev || max_pts <= 0)
    return fail(ICT_ERR_BAD_ARG, "ict_tracker_set_points_dev: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  if (tracker_reserve(tr, T, total_pts, st)) return ICT_ERR_CUDA;
  CU(cudaMemcpyAsync(tr->pt_off.p, pt_off_dev, sizeof(int64_t) * (size_t)(T + 1), cudaMemcpyDeviceToDevice, st));
  CU(launch_set_points(T, tr->pt_off.as<int64_t>(), pts_dev, nullptr, tr->pt3d.as<float>(), tr->norm.as<double>(),
                       tr->op.donorm, tr->op.maxpttrack, max_pts, st));
  tr->T = T;
  tr->total = total_pts;
  tr->max_pts = max_pts;
  tr->pts_maxpttrack = tr->op.maxpttrack;
  tr->pts_donorm = tr->op.donorm;
  tr->h_off.clear();
  tr->have_2d = false;
  tr->state_valid = false;
  return ICT_OK;
}

// k_set_points stores min(n, maxpttrack) points per track, normalised or not by donorm: a later optparam with another
// maxpttrack or donorm would make the kernels read points that were never stored, or undo a normalisation that does
// not match them.  Every call that reads the points refuses until ict_tracker_set_points runs again.
static int points_current(const ict_tracker* tr) {
  if (tr->T <= 0) return fail(ICT_ERR_BAD_ARG, "no points set: call ict_tracker_set_points first");
  if (tr->op.maxpttrack != tr->pts_maxpttrack || tr->op.donorm != tr->pts_donorm)
    return fail(ICT_ERR_BAD_ARG, "maxpttrack or donorm changed since the points were set: call ict_tracker_set_points "
                                 "again");
  return ICT_OK;
}

static TrackKernel tracker_kernel(const ict_tracker* tr, const ict_frames* fs) {
  return select_track_kernel(tr->op, tr->max_pts, tr->sum_mode, tr->eigen_packet, tr->force_general, tr->knob_no_k2r,
                             fs->tma_ok);
}

// SetPose + TrackPose for all tracks; every pointer is device memory.
static int run_tracks(ict_tracker* tr, const ict_frames* fs, const int* rf_dev, const int* nf_dev, int fixed_ref,
                      int fixed_new, const double* p_in_dev, double* p_out_dev, int* iters_dev, float* trace_dev,
                      int trace_cap, long long* npix_dev, cudaStream_t st) {
  if (!tr || !fs) return fail(ICT_ERR_BAD_ARG, "null tracker / frame store");
  if (points_current(tr)) return ICT_ERR_BAD_ARG;
  if (fs->lv_f != tr->op.lv_f || fs->pad != tr->op.psz || fs->w != tr->wh[0] || fs->h != tr->wh[1])
    return fail(ICT_ERR_BAD_ARG, "frame store does not match the tracker (need lv_f, pad == psz, w, h equal)");
  if (!rf_dev && (fixed_ref < 0 || fixed_ref >= fs->nframes || fixed_new < 0 || fixed_new >= fs->nframes))
    return fail(ICT_ERR_BAD_ARG, "frame index out of range");
  TrackParams prm;
  memset(&prm, 0, sizeof(prm));
  prm.op = tr->op;
  prm.cam = tr->cam;
  prm.frames = fs->desc;
  prm.ref_frame = rf_dev;
  prm.new_frame = nf_dev;
  prm.fixed_ref = fixed_ref;
  prm.fixed_new = fixed_new;
  prm.pt_off = tr->pt_off.as<int64_t>();
  prm.pt3d = tr->pt3d.as<float>();
  prm.norm = tr->norm.as<double>();
  prm.p_in = p_in_dev;
  prm.p_out = p_out_dev;
  prm.iters = iters_dev;
  prm.trace = trace_dev;
  prm.trace_cap = trace_cap;
  prm.teacher = (trace_dev && tr->teacher_cap > 0 && tr->teacher_cap == trace_cap) ? tr->teacher.as<float>() : nullptr;
  prm.npixres = npix_dev;
  prm.pt2d_out = tr->pt2d.as<float>();
  prm.T = tr->T;
  prm.t0 = 0;
  prm.sum_mode = tr->sum_mode;
  prm.eigen_packet = tr->eigen_packet;
  prm.tma_ok = fs->tma_ok ? 1 : 0;
  prm.force_general = tr->force_general;
  prm.seq_n = tr->seq_n;
  prm.seq_step = tr->seq_step;
  prm.knob_no_k2r = tr->knob_no_k2r;
  prm.knob_seq_launches = tr->knob_seq_launches;
  prm.robust = tr->robust;
  const TrackKernel kern = tracker_kernel(tr, fs);
  if (tr->robust && kern != TrackKernel::V8)
    return fail(ICT_ERR_UNSUPPORTED, "robustness modes need the fast mode (sum order 0), psz 8 and at most 240 points per track");
  if (tr->keep_state) {
    // carried template state: implemented by the reference-order kernel for 8x8 patches (the drivers' configuration),
    // with either packet width (the carried template does not depend on the order of the sums)
    if (kern != TrackKernel::X8 || tr->op.psz != 8)
      return fail(ICT_ERR_UNSUPPORTED, "keep_state needs the reference summation order, psz 8 and at most 224 points per track");
    const int P = tr->max_pts < tr->op.maxpttrack ? tr->max_pts : tr->op.maxpttrack;
    prm.state_stride = (int64_t)(3 * 64 + 12) * P;
    const size_t bytes = sizeof(float) * (size_t)prm.state_stride * tr->T;
    if (tr->state.cap < bytes) tr->state_valid = false;
    CU(tr->state.reserve(bytes));
    prm.state = tr->state.as<float>();
    prm.state_load = tr->state_valid ? 1 : 0;
  }
  if (kern != TrackKernel::MultiCta) {
    CU(launch_track(prm, tr->max_pts, st));
  } else {
    // tracks too large for one CTA's shared memory: multi-CTA path, one track at a time
    if (tr->h_off.empty()) return fail(ICT_ERR_UNSUPPORTED, "big tracks need host-side pt_off (use ict_tracker_set_points)");
    if (rf_dev) return fail(ICT_ERR_UNSUPPORTED, "big tracks take fixed ref/new frames (use ict_track_sequence or T=1)");
    size_t wb = 0;                          // work buffers sized for the largest track, reused in stream order
    for (int t = 0; t < tr->T; ++t) {
      const size_t w = bigtrack_work_bytes(tr->op, tr->h_off[t + 1] - tr->h_off[t], tr->eigen_packet);
      wb = w > wb ? w : wb;
    }
    // lanes: as many as there are tracks, at most ICT_BIG_LANES, and only while their work buffers stay below 2 GB
    int nl = tr->T < ict_tracker::ICT_BIG_LANES ? tr->T : ict_tracker::ICT_BIG_LANES;
    while (nl > 1 && wb * (size_t)nl > ((size_t)2 << 30)) --nl;
    if (nl <= 1) {
      CU(tr->big.reserve(wb));
      for (int t = 0; t < tr->T; ++t) {
        const int64_t n = tr->h_off[t + 1] - tr->h_off[t];
        if (tr->big_rf) { prm.fixed_ref = tr->big_rf[t]; prm.fixed_new = tr->big_nf[t]; }
        CU(launch_track_big(prm, t, n, tr->big.p, st));
      }
    } else {
      for (int k = 0; k < nl; ++k) {
        if (!tr->big_st[k]) CU(cudaStreamCreateWithFlags(&tr->big_st[k], cudaStreamNonBlocking));
        CU(tr->big_lane[k].reserve(wb));
      }
      for (int k = 0; k <= nl; ++k)
        if (!tr->big_ev[k]) CU(cudaEventCreateWithFlags(&tr->big_ev[k], cudaEventDisableTiming));
      CU(cudaEventRecord(tr->big_ev[nl], st));                 // the lanes start after what is already on the caller's stream
      for (int k = 0; k < nl; ++k) CU(cudaStreamWaitEvent(tr->big_st[k], tr->big_ev[nl], 0));
      for (int t = 0; t < tr->T; ++t) {
        const int k = t % nl;
        const int64_t n = tr->h_off[t + 1] - tr->h_off[t];
        if (tr->big_rf) { prm.fixed_ref = tr->big_rf[t]; prm.fixed_new = tr->big_nf[t]; }
        CU(launch_track_big(prm, t, n, tr->big_lane[k].p, tr->big_st[k]));
      }
      for (int k = 0; k < nl; ++k) {                            // ... and the caller's stream continues after all of them
        CU(cudaEventRecord(tr->big_ev[k], tr->big_st[k]));
        CU(cudaStreamWaitEvent(st, tr->big_ev[k], 0));
      }
    }
  }
  tr->have_2d = true;
  if (tr->keep_state) tr->state_valid = true;
  return ICT_OK;
}

int ict_track_batch_dev(ict_tracker* tr, const ict_frames* fs, const int* ref_frame_dev, const int* new_frame_dev,
                        const double* p_in_dev, double* p_out_dev, int* iters_dev, float* trace_dev, int trace_cap,
                        int64_t* npixres_dev, void* stream) {
  if (!ref_frame_dev || !new_frame_dev || !p_in_dev || !p_out_dev) return fail(ICT_ERR_BAD_ARG, "null device pointer");
  return run_tracks(tr, fs, ref_frame_dev, new_frame_dev, -1, -1, p_in_dev, p_out_dev, iters_dev, trace_dev,
                    trace_dev ? trace_cap : 0, (long long*)npixres_dev, (cudaStream_t)stream);
}

int ict_track_batch(ict_tracker* tr, const ict_frames* fs, const int* ref_frame, const int* new_frame,
                    const double* p_in, double* p_out, int* iters, float* trace, int trace_cap, int64_t* npixres) {
  if (!tr || !fs || !ref_frame || !new_frame || !p_in || !p_out) return fail(ICT_ERR_BAD_ARG, "null argument");
  const int T = tr->T;
  if (points_current(tr)) return ICT_ERR_BAD_ARG;
  const int L = tr->op.lv_f - tr->op.lv_l + 1;
  for (int t = 0; t < T; ++t)
    if (ref_frame[t] < 0 || ref_frame[t] >= fs->nframes || new_frame[t] < 0 || new_frame[t] >= fs->nframes)
      return fail(ICT_ERR_BAD_ARG, "frame index out of range");
  CU(tr->rf.reserve(sizeof(int) * (size_t)T));
  CU(tr->nf.reserve(sizeof(int) * (size_t)T));
  CU(tr->p_in.reserve(sizeof(double) * 6 * (size_t)T));
  CU(tr->p_out.reserve(sizeof(double) * 6 * (size_t)T));
  CU(tr->iters.reserve(sizeof(int) * (size_t)T * L));
  CU(tr->npix.reserve(sizeof(long long) * (size_t)T));
  if (trace && trace_cap > 0) CU(tr->trace.reserve(sizeof(float) * ICT_TRACE_FLOATS * (size_t)T * trace_cap));
  CU(cudaMemcpyAsync(tr->rf.p, ref_frame, sizeof(int) * (size_t)T, cudaMemcpyHostToDevice, 0));
  CU(cudaMemcpyAsync(tr->nf.p, new_frame, sizeof(int) * (size_t)T, cudaMemcpyHostToDevice, 0));
  CU(cudaMemcpyAsync(tr->p_in.p, p_in, sizeof(double) * 6 * (size_t)T, cudaMemcpyHostToDevice, 0));
  const bool big = tracker_kernel(tr, fs) == TrackKernel::MultiCta;
  int rc;
  if (big) {
    // multi-CTA path: the tracks run one after the other on the stream, each with its own frame pair
    tr->big_rf = ref_frame;
    tr->big_nf = new_frame;
    rc = run_tracks(tr, fs, nullptr, nullptr, ref_frame[0], new_frame[0], tr->p_in.as<double>(), tr->p_out.as<double>(),
                    tr->iters.as<int>(), trace && trace_cap > 0 ? tr->trace.as<float>() : nullptr, trace_cap,
                    tr->npix.as<long long>(), 0);
    tr->big_rf = tr->big_nf = nullptr;
  } else {
    rc = run_tracks(tr, fs, tr->rf.as<int>(), tr->nf.as<int>(), -1, -1, tr->p_in.as<double>(), tr->p_out.as<double>(),
                    tr->iters.as<int>(), trace && trace_cap > 0 ? tr->trace.as<float>() : nullptr, trace_cap,
                    tr->npix.as<long long>(), 0);
  }
  if (rc) return rc;
  CU(cudaMemcpyAsync(p_out, tr->p_out.p, sizeof(double) * 6 * (size_t)T, cudaMemcpyDeviceToHost, 0));
  if (iters) CU(cudaMemcpyAsync(iters, tr->iters.p, sizeof(int) * (size_t)T * L, cudaMemcpyDeviceToHost, 0));
  if (npixres) CU(cudaMemcpyAsync(npixres, tr->npix.p, sizeof(long long) * (size_t)T, cudaMemcpyDeviceToHost, 0));
  if (trace && trace_cap > 0)
    CU(cudaMemcpyAsync(trace, tr->trace.p, sizeof(float) * ICT_TRACE_FLOATS * (size_t)T * trace_cap,
                       cudaMemcpyDeviceToHost, 0));
  CU(cudaStreamSynchronize(0));
  return ICT_OK;
}

int ict_track_batch_stream(ict_tracker* tr, const ict_frames* fs, const int* ref_frame, const int* new_frame,
                           const double* p_in, double* p_out, int* iters, int64_t* npixres, void* stream) {
  if (!tr || !fs || !ref_frame || !new_frame || !p_in || !p_out) return fail(ICT_ERR_BAD_ARG, "null argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int T = tr->T;
  if (points_current(tr)) return ICT_ERR_BAD_ARG;
  if (tracker_kernel(tr, fs) == TrackKernel::MultiCta)
    return fail(ICT_ERR_UNSUPPORTED, "stream variant handles tracks that fit one CTA");
  for (int t = 0; t < T; ++t)
    if (ref_frame[t] < 0 || ref_frame[t] >= fs->nframes || new_frame[t] < 0 || new_frame[t] >= fs->nframes)
      return fail(ICT_ERR_BAD_ARG, "frame index out of range");
  const int L = tr->op.lv_f - tr->op.lv_l + 1;
  CU(tr->rf.reserve(sizeof(int) * (size_t)T));
  CU(tr->nf.reserve(sizeof(int) * (size_t)T));
  CU(tr->p_in.reserve(sizeof(double) * 6 * (size_t)T));
  CU(tr->p_out.reserve(sizeof(double) * 6 * (size_t)T));
  CU(tr->iters.reserve(sizeof(int) * (size_t)T * L));
  CU(tr->npix.reserve(sizeof(long long) * (size_t)T));
  CU(tr->lane_in.begin());
  CU(cudaMemcpyAsync(tr->rf.p, ref_frame, sizeof(int) * (size_t)T, cudaMemcpyHostToDevice, tr->lane_in.s));
  CU(cudaMemcpyAsync(tr->nf.p, new_frame, sizeof(int) * (size_t)T, cudaMemcpyHostToDevice, tr->lane_in.s));
  CU(cudaMemcpyAsync(tr->p_in.p, p_in, sizeof(double) * 6 * (size_t)T, cudaMemcpyHostToDevice, tr->lane_in.s));
  CU(tr->lane_in.publish(st));
  const int rc = run_tracks(tr, fs, tr->rf.as<int>(), tr->nf.as<int>(), -1, -1, tr->p_in.as<double>(),
                            tr->p_out.as<double>(), tr->iters.as<int>(), nullptr, 0, tr->npix.as<long long>(), st);
  if (rc) return rc;
  CU(tr->lane.done(st));
  CU(tr->lane_in.done(st));
  CU(cudaMemcpyAsync(p_out, tr->p_out.p, sizeof(double) * 6 * (size_t)T, cudaMemcpyDeviceToHost, st));
  if (iters) CU(cudaMemcpyAsync(iters, tr->iters.p, sizeof(int) * (size_t)T * L, cudaMemcpyDeviceToHost, st));
  if (npixres) CU(cudaMemcpyAsync(npixres, tr->npix.p, sizeof(long long) * (size_t)T, cudaMemcpyDeviceToHost, st));
  return ICT_OK;
}

int ict_track_sequence(ict_tracker* tr, const ict_frames* fs, int first, int nsteps, int step, const double* p_in,
                       double* poses_out, int* iters, int64_t* npixres) {
  if (!tr || !fs || !p_in || !poses_out || nsteps < 0 || (step != 1 && step != -1))
    return fail(ICT_ERR_BAD_ARG, "ict_track_sequence: bad argument");
  const int T = tr->T;
  if (points_current(tr)) return ICT_ERR_BAD_ARG;
  const int L = tr->op.lv_f - tr->op.lv_l + 1;
  const int last = first + nsteps * step;
  if (first < 0 || first >= fs->nframes || last < 0 || last >= fs->nframes)
    return fail(ICT_ERR_BAD_ARG, "frame range out of bounds");
  // all poses of the chain live on the device: the output of step k is the input of step k+1
  CU(tr->p_out.reserve(sizeof(double) * 6 * (size_t)T * (nsteps + 1)));
  CU(tr->iters.reserve(sizeof(int) * (size_t)T * L * (nsteps ? nsteps : 1)));
  CU(tr->npix.reserve(sizeof(long long) * (size_t)T * (nsteps ? nsteps : 1)));
  double* chain = tr->p_out.as<double>();
  CU(cudaMemcpyAsync(chain, p_in, sizeof(double) * 6 * (size_t)T, cudaMemcpyHostToDevice, 0));
  if (nsteps > 1 && tracker_kernel(tr, fs) == TrackKernel::V8 && !tr->knob_seq_launches) {
    // K2v8 loops over the frames inside the kernel: one launch for the whole chain
    tr->seq_n = nsteps;
    tr->seq_step = step;
    int rc = run_tracks(tr, fs, nullptr, nullptr, first, first + step, chain, chain + (size_t)6 * T, tr->iters.as<int>(),
                        nullptr, 0, tr->npix.as<long long>(), 0);
    tr->seq_n = tr->seq_step = 0;
    if (rc) return rc;
  } else {
    for (int k = 0; k < nsteps; ++k) {
      const int fr = first + k * step;
      int rc = run_tracks(tr, fs, nullptr, nullptr, fr, fr + step, chain + (size_t)k * 6 * T,
                          chain + (size_t)(k + 1) * 6 * T, tr->iters.as<int>() + (size_t)k * T * L, nullptr, 0,
                          tr->npix.as<long long>() + (size_t)k * T, 0);
      if (rc) return rc;
    }
  }
  CU(cudaMemcpyAsync(poses_out, chain, sizeof(double) * 6 * (size_t)T * (nsteps + 1), cudaMemcpyDeviceToHost, 0));
  if (iters && nsteps)
    CU(cudaMemcpyAsync(iters, tr->iters.p, sizeof(int) * (size_t)T * L * nsteps, cudaMemcpyDeviceToHost, 0));
  if (npixres && nsteps)
    CU(cudaMemcpyAsync(npixres, tr->npix.p, sizeof(long long) * (size_t)T * nsteps, cudaMemcpyDeviceToHost, 0));
  CU(cudaStreamSynchronize(0));
  return ICT_OK;
}

int ict_tracker_reproject(ict_tracker* tr, const double* p_in, float* pt2d_out) {
  if (!tr || !p_in) return fail(ICT_ERR_BAD_ARG, "null argument");
  if (points_current(tr)) return ICT_ERR_BAD_ARG;
  CU(tr->p_in.reserve(sizeof(double) * 6 * (size_t)tr->T));
  CU(cudaMemcpyAsync(tr->p_in.p, p_in, sizeof(double) * 6 * (size_t)tr->T, cudaMemcpyHostToDevice, 0));
  TrackParams prm;
  memset(&prm, 0, sizeof(prm));
  prm.op = tr->op;
  prm.cam = tr->cam;
  prm.pt_off = tr->pt_off.as<int64_t>();
  prm.pt3d = tr->pt3d.as<float>();
  prm.norm = tr->norm.as<double>();
  prm.p_in = tr->p_in.as<double>();
  prm.pt2d_out = tr->pt2d.as<float>();
  prm.T = tr->T;
  CU(launch_reproject(prm, 0));
  tr->have_2d = true;
  if (pt2d_out) CU(cudaMemcpy(pt2d_out, tr->pt2d.p, sizeof(float) * 2 * (size_t)tr->total, cudaMemcpyDeviceToHost));
  return ICT_OK;
}

int ict_tracker_get_2dpoints(ict_tracker* tr, float* out) {
  if (!tr || !out) return fail(ICT_ERR_BAD_ARG, "null argument");
  if (points_current(tr)) return ICT_ERR_BAD_ARG;
  if (!tr->have_2d) return fail(ICT_ERR_BAD_ARG, "no SetPose has run yet");
  CU(cudaMemcpy(out, tr->pt2d.p, sizeof(float) * 2 * (size_t)tr->total, cudaMemcpyDeviceToHost));
  return ICT_OK;
}

int ict_track_pair(const ict_optparam* op, const float fc[2], const float cc[2], const int wh[2], const float* imgA,
                   const float* imgB, double* pt3d, int npts, const double p_in[6], double p_out[6], int* iters,
                   float* trace, int trace_cap) {
  if (require_device()) return ICT_ERR_NO_DEVICE;
  if (!op || !imgA || !imgB || !pt3d || npts <= 0) return fail(ICT_ERR_BAD_ARG, "ict_track_pair: bad argument");
  ict_frames* fs = ict_frames_create(2, wh[0], wh[1], op->lv_f, op->psz);
  if (!fs) return ICT_ERR_BAD_ARG;
  ict_tracker* tr = ict_tracker_create(op, fc, cc, wh);
  int rc = tr ? ICT_OK : ICT_ERR_BAD_ARG;
  if (rc == ICT_OK) rc = ict_frames_upload(fs, 0, 1, imgA);
  if (rc == ICT_OK) rc = ict_frames_upload(fs, 1, 1, imgB);
  const int64_t off[2] = {0, npts};
  if (rc == ICT_OK) rc = ict_tracker_set_points(tr, 1, off, pt3d, 1);
  const int rf = 0, nf = 1;
  if (rc == ICT_OK) rc = ict_track_batch(tr, fs, &rf, &nf, p_in, p_out, iters, trace, trace_cap, nullptr);
  ict_tracker_destroy(tr);
  ict_frames_destroy(fs);
  return rc;
}

int ict_pose_hypotheses(const float fc[2], const float cc[2], int npts, const double* pt2d, const double* pt3d, int nsamples,
                        const int* sample_idx, const double p_init[6], double inlthresh, int maxiter, double* out_pose,
                        int* out_status, int* out_ninl, unsigned char* out_inlmask) {
  if (require_device()) return ICT_ERR_NO_DEVICE;
  if (!fc || !cc || !pt2d || !pt3d || !sample_idx || !p_init || !out_pose || !out_status || npts < 4 || nsamples < 0 ||
      !(inlthresh > 0) || maxiter < 1)
    return fail(ICT_ERR_BAD_ARG, "ict_pose_hypotheses: bad argument");
  if (nsamples == 0) return ICT_OK;
  DevBuf d2, d3, ds, dp, dst, dn, dm;
  cudaError_t e = d2.reserve(sizeof(double) * 2 * npts);
  if (e == cudaSuccess) e = d3.reserve(sizeof(double) * 3 * npts);
  if (e == cudaSuccess) e = ds.reserve(sizeof(int) * 4 * (size_t)nsamples);
  if (e == cudaSuccess) e = dp.reserve(sizeof(double) * 6 * (size_t)nsamples);
  if (e == cudaSuccess) e = dst.reserve(sizeof(int) * (size_t)nsamples);
  if (e == cudaSuccess) e = dn.reserve(sizeof(int) * (size_t)nsamples);
  if (e == cudaSuccess) e = dm.reserve((size_t)nsamples * npts);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d2.p, pt2d, sizeof(double) * 2 * npts, cudaMemcpyHostToDevice, 0);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d3.p, pt3d, sizeof(double) * 3 * npts, cudaMemcpyHostToDevice, 0);
  if (e == cudaSuccess) e = cudaMemcpyAsync(ds.p, sample_idx, sizeof(int) * 4 * (size_t)nsamples, cudaMemcpyHostToDevice, 0);
  const double fcd[2] = {fc[0], fc[1]}, ccd[2] = {cc[0], cc[1]};
  if (e == cudaSuccess)
    e = launch_hypotheses(fcd, ccd, npts, d2.as<double>(), d3.as<double>(), nsamples, ds.as<int>(), p_init, inlthresh, maxiter,
                          dp.as<double>(), dst.as<int>(), dn.as<int>(), dm.as<unsigned char>(), 0);
  if (e == cudaSuccess) e = cudaMemcpyAsync(out_pose, dp.p, sizeof(double) * 6 * (size_t)nsamples, cudaMemcpyDeviceToHost, 0);
  if (e == cudaSuccess) e = cudaMemcpyAsync(out_status, dst.p, sizeof(int) * (size_t)nsamples, cudaMemcpyDeviceToHost, 0);
  if (e == cudaSuccess && out_ninl) e = cudaMemcpyAsync(out_ninl, dn.p, sizeof(int) * (size_t)nsamples, cudaMemcpyDeviceToHost, 0);
  if (e == cudaSuccess && out_inlmask) e = cudaMemcpyAsync(out_inlmask, dm.p, (size_t)nsamples * npts, cudaMemcpyDeviceToHost, 0);
  if (e == cudaSuccess) e = cudaStreamSynchronize(0);
  int rc = ICT_OK;
  if (e != cudaSuccess) rc = fail(ICT_ERR_CUDA, std::string("ict_pose_hypotheses: ") + cudaGetErrorString(e));
  DevBuf* all[] = {&d2, &d3, &ds, &dp, &dst, &dn, &dm};
  for (DevBuf* b : all) b->release();
  return rc;
}

int ict_get_patches(const ict_frames* fs, int frame, int level, const ict_optparam* op, int npatch, const float* mids,
                    float* out_I, float* out_dx, float* out_dy) {
  if (!fs || !op || !mids || npatch < 0) return fail(ICT_ERR_BAD_ARG, "ict_get_patches: null argument");
  if (frames_range_ok(fs, frame, 1)) return ICT_ERR_BAD_ARG;
  if (fs->view || !fs->I) return fail(ICT_ERR_BAD_ARG, "ict_get_patches: needs a store that owns its pixels (not a view)");
  if (level < 0 || level > fs->lv_f) return fail(ICT_ERR_BAD_ARG, "ict_get_patches: level out of range");
  if (op->psz < 1 || op->psz > fs->pad) return fail(ICT_ERR_BAD_ARG, "ict_get_patches: psz must be 1..padding of the store");
  if (npatch == 0) return ICT_OK;
  // a centre must keep its (psz+1)^2 footprint inside the padded plane: |x| within the level's extent (odometer.cpp:273-275
  // tests [0, swo] x [0, sho] before it samples); anything else is refused instead of read out of bounds
  const float swo = (float)(fs->sw[level] - 2 * fs->pad), sho = (float)(fs->sh[level] - 2 * fs->pad);
  for (int i = 0; i < npatch; ++i)
    if (!(mids[2 * i] >= 0 && mids[2 * i + 1] >= 0 && mids[2 * i] <= swo && mids[2 * i + 1] <= sho))
      return fail(ICT_ERR_BAD_ARG, "ict_get_patches: a centre lies outside [0, swo] x [0, sho] of the level");
  const size_t n = (size_t)op->psz * op->psz, tot = n * npatch;
  DevBuf dm, dout;
  cudaError_t e = dm.reserve(sizeof(float) * 2 * npatch);
  if (e == cudaSuccess) e = dout.reserve(sizeof(float) * 3 * tot);
  float* o = dout.as<float>();
  if (e == cudaSuccess) e = cudaMemcpyAsync(dm.p, mids, sizeof(float) * 2 * npatch, cudaMemcpyHostToDevice, 0);
  const size_t po = (size_t)frame * fs->plane_floats + fs->level_off[level];
  if (e == cudaSuccess)
    e = launch_get_patches(fs->I + po, fs->dx + po, fs->dy + po, fs->sw[level], op->psz, op->psz / 2, op->dopatchnorm ? 1 : 0,
                           npatch, dm.as<float>(), out_I ? o : nullptr, out_dx ? o + tot : nullptr, out_dy ? o + 2 * tot : nullptr, 0);
  if (e == cudaSuccess && out_I) e = cudaMemcpyAsync(out_I, o, sizeof(float) * tot, cudaMemcpyDeviceToHost, 0);
  if (e == cudaSuccess && out_dx) e = cudaMemcpyAsync(out_dx, o + tot, sizeof(float) * tot, cudaMemcpyDeviceToHost, 0);
  if (e == cudaSuccess && out_dy) e = cudaMemcpyAsync(out_dy, o + 2 * tot, sizeof(float) * tot, cudaMemcpyDeviceToHost, 0);
  if (e == cudaSuccess) e = cudaStreamSynchronize(0);
  int rc = ICT_OK;
  if (e != cudaSuccess) rc = fail(ICT_ERR_CUDA, std::string("ict_get_patches: ") + cudaGetErrorString(e));
  dm.release();
  dout.release();
  return rc;
}

int ict_ncc_score(ict_tracker* tr, const ict_frames* fs, int frame_b, int frame_r, int frame_f, int nback, int nfwd,
                  const float* pt2d_back, const float* pt2d_refe, const float* pt2d_forw, float* out_corr) {
  if (!tr || !fs || !pt2d_back || !pt2d_refe || !pt2d_forw || !out_corr) return fail(ICT_ERR_BAD_ARG, "null argument");
  if (tr->T <= 0 || tr->h_off.empty()) return fail(ICT_ERR_BAD_ARG, "no points set");
  if (points_current(tr)) return ICT_ERR_BAD_ARG;
  if (fs->view || !fs->I) return fail(ICT_ERR_BAD_ARG, "ict_ncc_score: needs a store that owns its pixels (not a view)");
  if (fs->lv_f != tr->op.lv_f || fs->pad != tr->op.psz || fs->w != tr->wh[0] || fs->h != tr->wh[1])
    return fail(ICT_ERR_BAD_ARG, "frame store does not match the tracker (need lv_f, pad == psz, w, h equal)");
  if (nback < 0 || nfwd < 0 || nback + nfwd == 0) return fail(ICT_ERR_BAD_ARG, "ict_ncc_score: nback + nfwd must be positive");
  if (frames_range_ok(fs, frame_b, 1) || frames_range_ok(fs, frame_r, 1) || frames_range_ok(fs, frame_f, 1))
    return ICT_ERR_BAD_ARG;
  const size_t total = (size_t)tr->total;
  DevBuf in, out;
  int rc = ICT_OK;
  cudaError_t e = in.reserve(sizeof(float) * 6 * total);
  if (e == cudaSuccess) e = out.reserve(sizeof(float) * total);
  float* d = in.as<float>();
  if (e == cudaSuccess) e = cudaMemcpyAsync(d, pt2d_back, sizeof(float) * 2 * total, cudaMemcpyHostToDevice, 0);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d + 2 * total, pt2d_refe, sizeof(float) * 2 * total, cudaMemcpyHostToDevice, 0);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d + 4 * total, pt2d_forw, sizeof(float) * 2 * total, cudaMemcpyHostToDevice, 0);
  const int l = tr->op.lv_l;
  const size_t fo = (size_t)fs->plane_floats;
  if (e == cudaSuccess)
    e = launch_ncc(tr->op, tr->cam, fs->I + frame_b * fo + fs->level_off[l], fs->I + frame_r * fo + fs->level_off[l],
                   fs->I + frame_f * fo + fs->level_off[l], nback, nfwd, tr->pt_off.as<int64_t>(), tr->T, d, d + 2 * total,
                   d + 4 * total, out.as<float>(), 0);
  if (e == cudaSuccess) e = cudaMemcpy(out_corr, out.p, sizeof(float) * total, cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) rc = fail(ICT_ERR_CUDA, std::string("ict_ncc_score: ") + cudaGetErrorString(e));
  in.release();
  out.release();
  return rc;
}

}  // extern "C"
