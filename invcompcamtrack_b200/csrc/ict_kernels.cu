// ict_kernels.cu — hand-written sm_100a kernels of the inverse-compositional GN tracking path.
//
//   K0  k_pyr_level0 / k_pyr_levelN   util_constructpyramide        utilities.cpp:14-52
//   K1a k_set_points                  OdometerClass::Set3Dpoints    odometer.cpp:171-239
//   K2  k_track<PSZ,PN>               SetPose + TrackPose           odometer.cpp:241-426, pose.cpp, utilities.cpp:55-189
//
// Compiled with -fmad=false (see ict_device.cuh).  No tensor cores: the loop is a gather + streaming
// reduction (about 0.6 flop/B), see DESIGN.md.
#include "ict_kernels.cuh"
#include "ict_device.cuh"

#include <atomic>

namespace ict {

static std::atomic<long long> g_launches{0};
int64_t launch_count(int reset) {
  long long v = g_launches.load();
  if (reset) g_launches.store(0);
  return v;
}
void count_launch() { g_launches.fetch_add(1); }

// ==================================================================================================
// K0 — pyramid: per level one launch over the PADDED output plane of every frame in the batch.
//   level 0   : v = src                                    (clone + convertTo CV_32F, utilities.cpp:21,26)
//   level l>0 : v = ((a+b)+(c+d))*0.25 of level l-1        (cv::resize 1/2 INTER_LINEAR == area-fast, :24)
//   dx = v(x+1)-v(x-1), dy = v(y+1)-v(y-1), 0 on the first/last col/row (Sobel ksize 1, REFLECT_101, :30-31)
//   padding: replicate for I (:40), zero for dx/dy (:45-46)
// Each thread produces one padded output pixel; neighbouring values are re-read through L1/L2 (the whole
// level is a few MB).  Pure HBM streaming: 4 B read + 12 B written per padded pixel at level 0.
// ==================================================================================================
template <typename SrcT>
__global__ void __launch_bounds__(256) k_pyr_level0(const SrcT* __restrict__ src, int w, int h, int pad,
                                                    float* __restrict__ I, float* __restrict__ dx,
                                                    float* __restrict__ dy, int64_t plane_stride) {
  const int sw = w + 2 * pad, sh = h + 2 * pad;
  const int X = blockIdx.x * blockDim.x + threadIdx.x;
  const int Y = blockIdx.y * blockDim.y + threadIdx.y;
  if (X >= sw || Y >= sh) return;
  const SrcT* s = src + (int64_t)blockIdx.z * w * h;
  const int x = X - pad, y = Y - pad;
  const int xc = min(max(x, 0), w - 1), yc = min(max(y, 0), h - 1);
  const float v = (float)s[(int64_t)yc * w + xc];
  const bool inside = (x >= 0) & (x < w) & (y >= 0) & (y < h);
  float gx = 0.0f, gy = 0.0f;
  if (inside) {
    if (x > 0 && x < w - 1) gx = (float)s[(int64_t)y * w + x + 1] - (float)s[(int64_t)y * w + x - 1];
    if (y > 0 && y < h - 1) gy = (float)s[(int64_t)(y + 1) * w + x] - (float)s[(int64_t)(y - 1) * w + x];
  }
  const int64_t o = (int64_t)blockIdx.z * plane_stride + (int64_t)Y * sw + X;
  I[o] = v;
  dx[o] = gx;
  dy[o] = gy;
}

__device__ __forceinline__ float mean4(const float* __restrict__ Ip, int swp, int pad, int x, int y) {
  const float* r0 = Ip + (int64_t)(2 * y + pad) * swp + 2 * x + pad;
  const float2 a = make_float2(__ldg(r0), __ldg(r0 + 1));
  const float2 c = make_float2(__ldg(r0 + swp), __ldg(r0 + swp + 1));
  return ((a.x + a.y) + (c.x + c.y)) * 0.25f;
}

__global__ void __launch_bounds__(256) k_pyr_levelN(float* __restrict__ I, float* __restrict__ dx,
                                                    float* __restrict__ dy, int64_t plane_stride, int64_t off_prev,
                                                    int swp, int64_t off_cur, int lw, int lh, int pad) {
  const int sw = lw + 2 * pad, sh = lh + 2 * pad;
  const int X = blockIdx.x * blockDim.x + threadIdx.x;
  const int Y = blockIdx.y * blockDim.y + threadIdx.y;
  if (X >= sw || Y >= sh) return;
  const float* Ip = I + (int64_t)blockIdx.z * plane_stride + off_prev;
  const int x = X - pad, y = Y - pad;
  const int xc = min(max(x, 0), lw - 1), yc = min(max(y, 0), lh - 1);
  const float v = mean4(Ip, swp, pad, xc, yc);
  const bool inside = (x >= 0) & (x < lw) & (y >= 0) & (y < lh);
  float gx = 0.0f, gy = 0.0f;
  if (inside) {
    if (x > 0 && x < lw - 1) gx = mean4(Ip, swp, pad, x + 1, y) - mean4(Ip, swp, pad, x - 1, y);
    if (y > 0 && y < lh - 1) gy = mean4(Ip, swp, pad, x, y + 1) - mean4(Ip, swp, pad, x, y - 1);
  }
  const int64_t o = (int64_t)blockIdx.z * plane_stride + off_cur + (int64_t)Y * sw + X;
  I[o] = v;
  dx[o] = gx;
  dy[o] = gy;
}

// ---- vectorised forms (4 output pixels per thread, 128-bit stores) ---------------------------------------------
// Used when the padded row length, the padding and every level width are multiples of 4, so that a group of four
// output pixels never straddles the image border and all vector accesses are 16-byte aligned.  Same arithmetic.
__device__ __forceinline__ void ld4(const float* p, float* v) {
  const float4 t = __ldg(reinterpret_cast<const float4*>(p));
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
__device__ __forceinline__ void ld4(const unsigned char* p, float* v) {
  const uchar4 t = __ldg(reinterpret_cast<const uchar4*>(p));
  v[0] = (float)t.x; v[1] = (float)t.y; v[2] = (float)t.z; v[3] = (float)t.w;
}

template <typename SrcT>
__global__ void __launch_bounds__(256) k_pyr_level0_v4(const SrcT* __restrict__ src, int w, int h, int pad,
                                                       float* __restrict__ I, float* __restrict__ dx,
                                                       float* __restrict__ dy, int64_t plane_stride) {
  const int sw = w + 2 * pad, sh = h + 2 * pad;
  const int X = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  const int Y = blockIdx.y * blockDim.y + threadIdx.y;
  if (X >= sw || Y >= sh) return;
  const SrcT* s = src + (int64_t)blockIdx.z * w * h;
  const int x = X - pad, y = Y - pad;
  const int yc = min(max(y, 0), h - 1);
  const bool yin = (y >= 0) & (y < h);
  float vi[4], gx[4] = {0.f, 0.f, 0.f, 0.f}, gy[4] = {0.f, 0.f, 0.f, 0.f};
  if (x < 0 || x >= w) {   // whole group in the left / right padding: replicate for I, zero gradients
    const float e = (float)s[(int64_t)yc * w + (x < 0 ? 0 : w - 1)];
    vi[0] = vi[1] = vi[2] = vi[3] = e;
  } else {
    const SrcT* row = s + (int64_t)yc * w + x;
    ld4(row, vi);
    if (yin) {
      const float left = x > 0 ? (float)row[-1] : 0.0f, right = x + 4 < w ? (float)row[4] : 0.0f;
      gx[0] = x > 0 ? vi[1] - left : 0.0f;
      gx[1] = vi[2] - vi[0];
      gx[2] = vi[3] - vi[1];
      gx[3] = x + 4 < w ? right - vi[2] : 0.0f;
      if (y > 0 && y < h - 1) {
        float up[4], dn[4];
        ld4(row - w, up);
        ld4(row + w, dn);
#pragma unroll
        for (int k = 0; k < 4; ++k) gy[k] = dn[k] - up[k];
      }
    }
  }
  const int64_t o = (int64_t)blockIdx.z * plane_stride + (int64_t)Y * sw + X;
  *reinterpret_cast<float4*>(I + o) = make_float4(vi[0], vi[1], vi[2], vi[3]);
  *reinterpret_cast<float4*>(dx + o) = make_float4(gx[0], gx[1], gx[2], gx[3]);
  *reinterpret_cast<float4*>(dy + o) = make_float4(gy[0], gy[1], gy[2], gy[3]);
}

// four 2x2 means of level l-1 at level-l columns x..x+3 (x multiple of 4), row y: two aligned float4 per source row
__device__ __forceinline__ void mean4x4(const float* __restrict__ Ip, int swp, int pad, int x, int y, float* v) {
  const float* r0 = Ip + (int64_t)(2 * y + pad) * swp + 2 * x + pad;
  float a[8], c[8];
  ld4(r0, a); ld4(r0 + 4, a + 4);
  ld4(r0 + swp, c); ld4(r0 + swp + 4, c + 4);
#pragma unroll
  for (int k = 0; k < 4; ++k) v[k] = ((a[2 * k] + a[2 * k + 1]) + (c[2 * k] + c[2 * k + 1])) * 0.25f;
}

__global__ void __launch_bounds__(256) k_pyr_levelN_v4(float* __restrict__ I, float* __restrict__ dx,
                                                       float* __restrict__ dy, int64_t plane_stride, int64_t off_prev,
                                                       int swp, int64_t off_cur, int lw, int lh, int pad) {
  const int sw = lw + 2 * pad, sh = lh + 2 * pad;
  const int X = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  const int Y = blockIdx.y * blockDim.y + threadIdx.y;
  if (X >= sw || Y >= sh) return;
  const float* Ip = I + (int64_t)blockIdx.z * plane_stride + off_prev;
  const int x = X - pad, y = Y - pad;
  const int yc = min(max(y, 0), lh - 1);
  const bool yin = (y >= 0) & (y < lh);
  float vi[4], gx[4] = {0.f, 0.f, 0.f, 0.f}, gy[4] = {0.f, 0.f, 0.f, 0.f};
  if (x < 0 || x >= lw) {
    const float e = mean4(Ip, swp, pad, x < 0 ? 0 : lw - 1, yc);
    vi[0] = vi[1] = vi[2] = vi[3] = e;
  } else {
    mean4x4(Ip, swp, pad, x, yc, vi);
    if (yin) {
      gx[0] = x > 0 ? vi[1] - mean4(Ip, swp, pad, x - 1, y) : 0.0f;
      gx[1] = vi[2] - vi[0];
      gx[2] = vi[3] - vi[1];
      gx[3] = x + 4 < lw ? mean4(Ip, swp, pad, x + 4, y) - vi[2] : 0.0f;
      if (y > 0 && y < lh - 1) {
        float up[4], dn[4];
        mean4x4(Ip, swp, pad, x, y - 1, up);
        mean4x4(Ip, swp, pad, x, y + 1, dn);
#pragma unroll
        for (int k = 0; k < 4; ++k) gy[k] = dn[k] - up[k];
      }
    }
  }
  const int64_t o = (int64_t)blockIdx.z * plane_stride + off_cur + (int64_t)Y * sw + X;
  *reinterpret_cast<float4*>(I + o) = make_float4(vi[0], vi[1], vi[2], vi[3]);
  *reinterpret_cast<float4*>(dx + o) = make_float4(gx[0], gx[1], gx[2], gx[3]);
  *reinterpret_cast<float4*>(dy + o) = make_float4(gy[0], gy[1], gy[2], gy[3]);
}

cudaError_t launch_pyramid(const float* src_f32, const unsigned char* src_u8, int count, int w, int h, int lv_f,
                           int pad, float* I, float* dx, float* dy, int64_t plane_floats,
                           const int64_t* level_off, cudaStream_t stream) {
  if (count <= 0) return cudaSuccess;
  const dim3 blk(32, 8, 1);
  // vector path: every level width, the padding and the image base addresses allow aligned groups of four
  const bool vec = (pad % 4 == 0) && ((w >> lv_f) % 4 == 0) && (plane_floats % 4 == 0) &&
                   (((uintptr_t)I | (uintptr_t)dx | (uintptr_t)dy) % 16 == 0) &&
                   (src_u8 ? ((uintptr_t)src_u8 % 4 == 0) : ((uintptr_t)src_f32 % 16 == 0));
  for (int z0 = 0; z0 < count; z0 += 65535) {
    const int zc = min(count - z0, 65535);
    float* Iz = I + (int64_t)z0 * plane_floats;
    float* dxz = dx + (int64_t)z0 * plane_floats;
    float* dyz = dy + (int64_t)z0 * plane_floats;
    {
      const int sw = w + 2 * pad, sh = h + 2 * pad;
      if (vec) {
        const dim3 grd((sw / 4 + 31) / 32, (sh + 7) / 8, zc);
        if (src_u8)
          k_pyr_level0_v4<unsigned char><<<grd, blk, 0, stream>>>(src_u8 + (int64_t)z0 * w * h, w, h, pad, Iz, dxz, dyz,
                                                                   plane_floats);
        else
          k_pyr_level0_v4<float><<<grd, blk, 0, stream>>>(src_f32 + (int64_t)z0 * w * h, w, h, pad, Iz, dxz, dyz,
                                                           plane_floats);
      } else {
        const dim3 grd((sw + 31) / 32, (sh + 7) / 8, zc);
        if (src_u8)
          k_pyr_level0<unsigned char><<<grd, blk, 0, stream>>>(src_u8 + (int64_t)z0 * w * h, w, h, pad, Iz, dxz, dyz,
                                                                plane_floats);
        else
          k_pyr_level0<float><<<grd, blk, 0, stream>>>(src_f32 + (int64_t)z0 * w * h, w, h, pad, Iz, dxz, dyz,
                                                        plane_floats);
      }
      count_launch();
    }
    for (int l = 1; l <= lv_f; ++l) {
      const int lw = w >> l, lh = h >> l;
      const int sw = lw + 2 * pad, sh = lh + 2 * pad;
      if (vec) {
        const dim3 grd((sw / 4 + 31) / 32, (sh + 7) / 8, zc);
        k_pyr_levelN_v4<<<grd, blk, 0, stream>>>(Iz, dxz, dyz, plane_floats, level_off[l - 1],
                                                 (w >> (l - 1)) + 2 * pad, level_off[l], lw, lh, pad);
      } else {
        const dim3 grd((sw + 31) / 32, (sh + 7) / 8, zc);
        k_pyr_levelN<<<grd, blk, 0, stream>>>(Iz, dxz, dyz, plane_floats, level_off[l - 1], (w >> (l - 1)) + 2 * pad,
                                              level_off[l], lw, lh, pad);
      }
      count_launch();
    }
  }
  return cudaGetLastError();
}

// ==================================================================================================
// K1a — Set3Dpoints (odometer.cpp:171-239): optional centring / division by the mean squared norm in
// fp64, then double -> float.  One CTA per track.  The fp64 sums run in the reference's sequential
// order on one thread for tracks up to SEQ_LIMIT points; longer tracks (dense alignment) use a fixed
// two-stage tree (fp64, so the difference is ~1e-16 relative and vanishes in the float cast).
// ==================================================================================================
#define ICT_SEQ_LIMIT 8192

__global__ void __launch_bounds__(256) k_set_points(int T, const int64_t* __restrict__ pt_off,
                                                    const double* pts, double* pts_mut,
                                                    float* __restrict__ pt3d, double* __restrict__ norm,
                                                    int donorm, int maxpttrack) {
  const int t = blockIdx.x;
  if (t >= T) return;
  const int64_t off = pt_off[t];
  const int n_in = (int)(pt_off[t + 1] - off);
  const int P = min(n_in, maxpttrack);
  const double* p1 = pts + 3 * off;
  const double* p2 = p1 + n_in;
  const double* p3 = p2 + n_in;
  float* q1 = pt3d + 3 * off;
  float* q2 = q1 + n_in;
  float* q3 = q2 + n_in;
  __shared__ double s_norm[4];
  __shared__ double s_red[3][8];
  const int tid = threadIdx.x, nt = blockDim.x;
  if (!donorm) {
    for (int i = tid; i < P; i += nt) {
      q1[i] = (float)p1[i];
      q2[i] = (float)p2[i];
      q3[i] = (float)p3[i];
    }
    if (tid < 4) norm[4 * (int64_t)t + tid] = 0.0;
    return;
  }
  if (P <= ICT_SEQ_LIMIT) {
    if (tid == 0) {
      const double nd = (double)P;
      double m0 = 0, m1 = 0, m2 = 0, var = 0;
      for (int i = 0; i < P; ++i) m0 += p1[i];
      for (int i = 0; i < P; ++i) m1 += p2[i];
      for (int i = 0; i < P; ++i) m2 += p3[i];
      m0 /= nd;
      m1 /= nd;
      m2 /= nd;
      for (int i = 0; i < P; ++i) {
        const double a = p1[i] - m0, b = p2[i] - m1, c = p3[i] - m2;
        var += a * a + b * b + c * c;
      }
      var /= nd;
      s_norm[0] = m0; s_norm[1] = m1; s_norm[2] = m2; s_norm[3] = var;
    }
  } else {
    // fixed-order tree: per-thread strided partials -> warp shuffle -> 8 warps
    double a[3] = {0, 0, 0};
    for (int i = tid; i < P; i += nt) { a[0] += p1[i]; a[1] += p2[i]; a[2] += p3[i]; }
    for (int k = 0; k < 3; ++k) {
      for (int o = 16; o > 0; o >>= 1) a[k] += __shfl_down_sync(0xffffffffu, a[k], o);
      if ((tid & 31) == 0) s_red[k][tid >> 5] = a[k];
    }
    __syncthreads();
    if (tid == 0)
      for (int k = 0; k < 3; ++k) {
        double s = 0;
        for (int wv = 0; wv < (nt >> 5); ++wv) s += s_red[k][wv];
        s_norm[k] = s / (double)P;
      }
    __syncthreads();
    double v = 0;
    for (int i = tid; i < P; i += nt) {
      const double x = p1[i] - s_norm[0], y = p2[i] - s_norm[1], z = p3[i] - s_norm[2];
      v += x * x + y * y + z * z;
    }
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((tid & 31) == 0) s_red[0][tid >> 5] = v;
    __syncthreads();
    if (tid == 0) {
      double s = 0;
      for (int wv = 0; wv < (nt >> 5); ++wv) s += s_red[0][wv];
      s_norm[3] = s / (double)P;
    }
  }
  __syncthreads();
  const double m0 = s_norm[0], m1 = s_norm[1], m2 = s_norm[2], var = s_norm[3];
  for (int i = tid; i < P; i += nt) {
    const double a = p1[i] - m0, b = p2[i] - m1, c = p3[i] - m2;
    q1[i] = (float)(a / var);
    q2[i] = (float)(b / var);
    q3[i] = (float)(c / var);
    if (pts_mut) {   // the reference centres the caller's array in place (odometer.cpp:207-212)
      pts_mut[3 * off + i] = a;
      pts_mut[3 * off + n_in + i] = b;
      pts_mut[3 * off + 2 * (int64_t)n_in + i] = c;
    }
  }
  if (tid < 4) norm[4 * (int64_t)t + tid] = s_norm[tid];
}

cudaError_t launch_set_points(int T, const int64_t* pt_off, const double* pts, double* pts_mut, float* pt3d,
                              double* norm, int donorm, int maxpttrack, int max_pts, cudaStream_t stream) {
  (void)max_pts;
  if (T <= 0) return cudaSuccess;
  k_set_points<<<T, 256, 0, stream>>>(T, pt_off, pts, pts_mut, pt3d, norm, donorm, maxpttrack);
  count_launch();
  return cudaGetLastError();
}

// ==================================================================================================
// K2 — SetPose + TrackPose, one CTA per track, all levels and iterations on device.
//
// Shared-memory residency: for every template pixel the CTA keeps (pat_ref, pat_dx, pat_dy) = 12 B
// in shared memory for the whole level; the six steepest-descent values are RECOMPUTED per iteration
// from (dx,dy) and ten per-point coefficients with exactly the reference's roundings
// (sd = fl(fl(dx*a)+fl(dy*b)), odometer.cpp:317-326), so they are bit-identical to the reference's
// stored sd arrays while cutting the per-pixel state from 28 B to 12 B.  The new frame is gathered
// with four read-only loads per pixel (weights constant per patch, utilities.cpp:65-76).
//
// Reference quirks preserved (SURVEY.md §9): ceil(x+1e-5f) placement, centre-only inclusive bounds
// test, stale template/SD of points that leave the reference image at a finer level (state is only
// zeroed at Set3Dpoints), new-frame-invisible points dropping out of J^T r but staying in H, min two
// iterations per level, additive se(3) update, intensity-only patch mean subtraction.
// ==================================================================================================
struct TrackShared {
  float G[12];
  float p[6];
  float Hsum[21];
  float part[32 * 21];
  Lu6 lu;
  float normdp, normdp_init;
  int cont, it, nvis;
  long long npix;
};

template <int PSZ>
__device__ __forceinline__ void elem_split(int e, int n, int psz, int& i, int& r, int& c) {
  if constexpr (PSZ > 0) {
    i = e / (PSZ * PSZ);
    const int rem = e - i * (PSZ * PSZ);
    r = rem / PSZ;
    c = rem - r * PSZ;
  } else {
    i = e / n;
    const int rem = e - i * n;
    r = rem / psz;
    c = rem - r * psz;
  }
}

// --------------------------------------------------------------------------------------------------
// Reference-order reductions (sum_mode 1).  Eigen's vectorised .sum() (Eigen 3.3 Redux.h, two packet accumulators —
// oracle/ictrack_oracle.c DEF_PACKET_SUM) is 2W interleaved SEQUENTIAL fp32 chains for W-float packets: chain c adds
// v[c], v[2W+c], v[4W+c], ... in that order — eight chains for SSE's 4-float packets (the default), sixteen for AVX's
// 8-float packets (TrackParams.eigen_packet == 8).  fp32 addition is not associative, so the only way to reproduce
// its bits is to run those chains as written: one thread per (quantity, chain), the other threads of the CTA idle.
// About 3x slower per iteration than the tree; exists so that parity with the reference can be shown BIT-EXACT and
// for callers who need reference-identical iteration counts.
// --------------------------------------------------------------------------------------------------
// mean of each visible patch of `buf` (n values per patch) -> s_mean[i]
template <bool EX, int W>
__device__ __forceinline__ void patch_means(const float* buf, float* s_mean, const int* s_vis, int visbit, int P,
                                            int n, int tid, int nt) {
  if (EX) {   // reference order, one thread per patch
    for (int i = tid; i < P; i += nt) {
      if (!(s_vis[i] & visbit)) continue;
      const float* b = buf + i * n;
      s_mean[i] = eigen_sum_serial<W>([&](int e) { return b[e]; }, n) / n;   // tmp.sum() / op->novals, utilities.cpp:112
    }
  } else {    // one warp per patch, lane-strided partials + shuffle tree
    const int lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
    for (int i = warp; i < P; i += nw) {
      if (!(s_vis[i] & visbit)) continue;
      float s = 0.0f;
      for (int k = lane; k < n; k += 32) s = s + buf[i * n + k];
      s = warp_sum(s);
      if (lane == 0) s_mean[i] = s / n;
    }
  }
}

// MODE bit 0: dopatchnorm; bit 1: reference-order (Eigen packet) sums.  Either one needs the fourth plane.
// Bit 2 (with bit 1): 8-float packets (sixteen chains) instead of 4-float ones (eight).
template <int PSZ, int MODE>
__global__ void __launch_bounds__(256) k_track(const TrackParams prm) {
  constexpr bool PN = (MODE & 1) != 0;
  constexpr bool EX = (MODE & 2) != 0;
  constexpr int PK = (MODE & 4) ? 8 : 4;              // Eigen packet width of the reference-order sums
  constexpr int NCH = 2 * PK;                         // chains per sum
  extern __shared__ __align__(16) float smem[];
  __shared__ TrackShared S;
  __shared__ float s_chain[21 * NCH];

  const int t = blockIdx.x + prm.t0;
  const ict_optparam& op = prm.op;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
  const int psz = PSZ > 0 ? PSZ : op.psz;
  const int n = PSZ > 0 ? PSZ * PSZ : op.novals;
  const int pszd2 = op.pszd2;
  const int64_t off = prm.pt_off[t];
  const int n_in = (int)(prm.pt_off[t + 1] - off);
  const int P = min(n_in, op.maxpttrack);
  const int E = P * n;
  const int Nfull = op.maxpttrack * n;               // the reference sums over ALL maxpttrack*novals slots
  const int Epad = (E + 3) & ~3;
  const bool donorm = op.donorm != 0;
  const bool patchnorm = PN && (op.dopatchnorm != 0);

  // ---- shared-memory carve-up ---------------------------------------------------------------------
  float* s_ref = smem;
  float* s_gx = s_ref + Epad;
  float* s_gy = s_gx + Epad;
  float* s_new = s_gy + Epad;                       // pat_new (PN) / pdiff (EX); absent when MODE == 0
  float* s_ptf = MODE ? s_new + Epad : s_new;       // per-point floats
  float* s_X = s_ptf;
  float* s_Y = s_X + P;
  float* s_Z = s_Y + P;
  float* s_Xc = s_Z + P;
  float* s_Yc = s_Xc + P;
  float* s_Zc = s_Yc + P;
  float* s_coef = s_Zc + P;                         // [10][P]
  float* s_w = s_coef + 10 * P;                     // [4][P]
  float* s_mean = s_w + 4 * P;                      // [P]
  int* s_base = (int*)(s_mean + P);                 // [P]
  int* s_vis = s_base + P;                          // [P] bit0: visible in ref (this level), bit1: in new

  const TrackFrames fr = track_frames(prm, t);

  // ---- ResetOdometer (odometer.cpp:580-609) + load float points ------------------------------------
  for (int e = tid; e < Epad; e += nt) { s_ref[e] = 0.0f; s_gx[e] = 0.0f; s_gy[e] = 0.0f; }
  {
    const float* q = prm.pt3d + 3 * off;
    for (int i = tid; i < P; i += nt) {
      s_X[i] = q[i];
      s_Y[i] = q[n_in + i];
      s_Z[i] = q[2 * (int64_t)n_in + i];
      s_vis[i] = 0;
#pragma unroll
      for (int k = 0; k < 10; ++k) s_coef[k * P + i] = 0.0f;
    }
  }
  // ---- SetPose: setpose_se3 (pose.cpp:25-76) ----------------------------------------------------------
  if (tid == 0) {
    track_setpose_from(prm, prm.p_in, t, donorm, S.p, S.G, S.Hsum);
    S.npix = 0;
    S.nvis = 0;
  }
  __syncthreads();
  // project_pt_save_rotated: camera-frame points frozen for the whole TrackPose
  for (int i = tid; i < P; i += nt) save_rotated_point(prm, S.Hsum, off, n_in, i, s_X[i], s_Y[i], s_Z[i], s_Xc, s_Yc, s_Zc);
  __syncthreads();

  float* trace = track_trace(prm, t);
  int trace_n = 0;   // thread 0 only

  // sd_q(e) with the reference's roundings, from shared memory (used by the reference-order chains)
  auto sd_at = [&](int q, int e) -> float {
    const int i = PSZ > 0 ? e / (PSZ * PSZ) : e / n;
    const float gx = s_gx[e], gy = s_gy[e];
    switch (q) {
      case 0: return gx * s_coef[0 * P + i];
      case 1: return gy * s_coef[1 * P + i];
      case 2: return gx * s_coef[2 * P + i] + gy * s_coef[3 * P + i];
      case 3: return gx * s_coef[4 * P + i] + gy * s_coef[5 * P + i];
      case 4: return gx * s_coef[6 * P + i] + gy * s_coef[7 * P + i];
      default: return gx * s_coef[8 * P + i] + gy * s_coef[9 * P + i];
    }
  };

  for (int sl = op.lv_f; sl >= op.lv_l; --sl) {
    const float fx = prm.cam.fx[sl], fy = prm.cam.fy[sl], cx = prm.cam.cx[sl], cy = prm.cam.cy[sl];
    const float swo = prm.cam.swo[sl], sho = prm.cam.sho[sl];
    const int width = prm.cam.width[sl];
    const float* __restrict__ Iref = fr.ref->I[sl];
    const float* __restrict__ Dxr = fr.ref->dx[sl];
    const float* __restrict__ Dyr = fr.ref->dy[sl];
    const float* __restrict__ Inew = fr.nw->I[sl];

    // ---- 4a. per point: reference placement + SD coefficients (odometer.cpp:268-279, 306-326) ---------
    for (int i = tid; i < P; i += nt) {
      const float xc = s_Xc[i], yc = s_Yc[i], zc = s_Zc[i];
      const float mx = (xc / zc) * fx + cx;      // pt2d[sl][i], project_pt at the pose set by SetPose
      const float my = (yc / zc) * fy + cy;
      // odometer.cpp:273-275; written so that a NaN centre counts as outside (the reference would index with it)
      const bool out = !((mx >= 0) & (my >= 0) & (mx <= swo) & (my <= sho));
      if (out) {
        s_vis[i] = 0;
      } else {
        s_vis[i] = 1;
        const PatchPlace q = patch_place(mx, my, pszd2, width);
        s_base[i] = q.base;
        s_w[i] = q.w0; s_w[P + i] = q.w1; s_w[2 * P + i] = q.w2; s_w[3 * P + i] = q.w3;
        float c[10];
        sd_coefs(xc, yc, zc, fx, fy, c);
#pragma unroll
        for (int k = 0; k < 10; ++k) s_coef[k * P + i] = c[k];
      }
    }
    __syncthreads();
    // ---- 4b. template gather: pat_ref, pat_dx, pat_dy (util_getPatch_grad, utilities.cpp:115-189) -----
    for (int e = tid; e < E; e += nt) {
      int i, r, c;
      elem_split<PSZ>(e, n, psz, i, r, c);
      if (s_vis[i] & 1) {
        const int addr = s_base[i] + r * width + c;
        const float w0 = s_w[i], w1 = s_w[P + i], w2 = s_w[2 * P + i], w3 = s_w[3 * P + i];
        s_ref[e] = bilin4(Iref, addr, width, w0, w1, w2, w3);
        s_gx[e] = bilin4(Dxr, addr, width, w0, w1, w2, w3);
        s_gy[e] = bilin4(Dyr, addr, width, w0, w1, w2, w3);
      }
    }
    if (patchnorm) {
      __syncthreads();
      patch_means<EX, PK>(s_ref, s_mean, s_vis, 1, P, n, tid, nt);
      __syncthreads();
      for (int e = tid; e < E; e += nt) {
        const int i = e / n;
        if (s_vis[i] & 1) s_ref[e] = s_ref[e] - s_mean[i];
      }
    }
    // ---- 5+6. steepest-descent values and Hessian (odometer.cpp:302-334, 428-472) ---------------------
    if (EX) {
      __syncthreads();
      const int as2 = (Nfull / NCH) * NCH;
      for (int qc = tid; qc < 21 * NCH; qc += nt) {    // 21 x 16 chains exceed the block: loop over (quantity, chain)
        const int q = qc / NCH, c = qc % NCH;
        int a = 0, b = 0, k = 0;                       // q-th pair (a<=b) in the order of ComputeHessian
        for (int aa = 0; aa < 6; ++aa)
          for (int bb = aa; bb < 6; ++bb) { if (k == q) { a = aa; b = bb; } ++k; }
        s_chain[qc] = eigen_chain<PK>([&](int e) { return sd_at(a, e) * sd_at(b, e); }, c, as2, E);
      }
      __syncthreads();
      if (tid < 21) {
        int a = 0, b = 0, k = 0;
        for (int aa = 0; aa < 6; ++aa)
          for (int bb = aa; bb < 6; ++bb) { if (k == tid) { a = aa; b = bb; } ++k; }
        S.Hsum[tid] = eigen_finish<PK>(s_chain + NCH * tid, [&](int e) { return sd_at(a, e) * sd_at(b, e); }, Nfull, E);
      }
    } else {
      float acc[21];
#pragma unroll
      for (int k = 0; k < 21; ++k) acc[k] = 0.0f;
      for (int e = tid; e < E; e += nt) {
        int i, r, c;
        elem_split<PSZ>(e, n, psz, i, r, c);
        float cf[10], sd[6];
#pragma unroll
        for (int k = 0; k < 10; ++k) cf[k] = s_coef[k * P + i];
        sd_values(s_gx[e], s_gy[e], cf, sd);
        int k = 0;
#pragma unroll
        for (int a = 0; a < 6; ++a)
#pragma unroll
          for (int b = a; b < 6; ++b) { acc[k] = acc[k] + sd[a] * sd[b]; ++k; }
      }
#pragma unroll
      for (int k = 0; k < 21; ++k) {
        const float v = warp_sum(acc[k]);
        if (lane == 0) S.part[warp * 21 + k] = v;
      }
      __syncthreads();
      if (tid < 21) {
        float s = S.part[tid];
        for (int wv = 1; wv < nw; ++wv) s = s + S.part[wv * 21 + tid];
        S.Hsum[tid] = s;
      }
    }
    __syncthreads();
    if (warp == 0) lu6_factor_warp(S.Hsum, S.lu);  // factor once; the solves below repeat Eigen's op order
    if (tid == 0) {
      S.normdp_init = 1e-10f;                      // odometer.cpp:341-342
      S.normdp = 1e-10f;
      S.it = 0;
      S.cont = keep_iterating(op, 0, 1e-10f, 1e-10f);
    }
    __syncthreads();

    // ---- iterations (odometer.cpp:344-419) -------------------------------------------------------------
    while (S.cont) {
      // 7. project_pt with the current pose (pose.cpp:307-397) + new-frame placement
      for (int i = tid; i < P; i += nt) {
        float tx, ty, tz;
        rigid_apply<float>(S.G, s_X[i], s_Y[i], s_Z[i], tx, ty, tz);
        const float mx = (tx / tz) * fx + cx;
        const float my = (ty / tz) * fy + cy;
        const bool out = !((mx >= 0) & (my >= 0) & (mx <= swo) & (my <= sho));   // odometer.cpp:369-371
        if (out) {
          s_vis[i] &= ~2;
        } else {
          s_vis[i] |= 2;
          const PatchPlace q = patch_place(mx, my, pszd2, width);
          s_base[i] = q.base;
          s_w[i] = q.w0; s_w[P + i] = q.w1; s_w[2 * P + i] = q.w2; s_w[3 * P + i] = q.w3;
          atomicAdd(&S.nvis, 1);
        }
      }
      __syncthreads();
      // 8. new-frame patch, residual, projection on the SD images
      if (patchnorm) {
        for (int e = tid; e < E; e += nt) {
          int i, r, c;
          elem_split<PSZ>(e, n, psz, i, r, c);
          if (s_vis[i] & 2)
            s_new[e] = bilin4(Inew, s_base[i] + r * width + c, width, s_w[i], s_w[P + i], s_w[2 * P + i],
                              s_w[3 * P + i]);
        }
        __syncthreads();
        patch_means<EX, PK>(s_new, s_mean, s_vis, 2, P, n, tid, nt);
        __syncthreads();
      }
      if (EX) {
        // pdiff of every slot (0 where the point is not visible: its sd_proj stays memset to 0, :352-357)
        for (int e = tid; e < E; e += nt) {
          int i, r, c;
          elem_split<PSZ>(e, n, psz, i, r, c);
          float pd = 0.0f;
          if (s_vis[i] & 2) {
            float pn;
            if (patchnorm)
              pn = s_new[e] - s_mean[i];
            else
              pn = bilin4(Inew, s_base[i] + r * width + c, width, s_w[i], s_w[P + i], s_w[2 * P + i], s_w[3 * P + i]);
            pd = s_ref[e] - pn;
          }
          s_new[e] = pd;
        }
        __syncthreads();
        const int as2 = (Nfull / NCH) * NCH;
        if (tid < 6 * NCH) {                           // 48 or 96 chains: the block has at least 192 threads
          const int q = tid / NCH, c = tid % NCH;
          s_chain[tid] = eigen_chain<PK>([&](int e) { return sd_at(q, e) * s_new[e]; }, c, as2, E);
        }
        __syncthreads();
        if (tid < 6)
          S.part[tid] = eigen_finish<PK>(s_chain + NCH * tid, [&](int e) { return sd_at(tid, e) * s_new[e]; }, Nfull, E);
      } else {
        float acc[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) acc[k] = 0.0f;
        for (int e = tid; e < E; e += nt) {
          int i, r, c;
          elem_split<PSZ>(e, n, psz, i, r, c);
          if (s_vis[i] & 2) {
            float pn;
            if (patchnorm)
              pn = s_new[e] - s_mean[i];
            else
              pn = bilin4(Inew, s_base[i] + r * width + c, width, s_w[i], s_w[P + i], s_w[2 * P + i], s_w[3 * P + i]);
            const float pd = s_ref[e] - pn;          // pdiff, odometer.cpp:381
            float cf[10], sd[6];
#pragma unroll
            for (int k = 0; k < 10; ++k) cf[k] = s_coef[k * P + i];
            sd_values(s_gx[e], s_gy[e], cf, sd);
#pragma unroll
            for (int k = 0; k < 6; ++k) acc[k] = acc[k] + sd[k] * pd;   // sd_k_proj then .sum(), :386-404
          }
        }
        // 9a. J^T r: warp shuffle tree, then fixed-order sum over warps
#pragma unroll
        for (int k = 0; k < 6; ++k) {
          const float v = warp_sum(acc[k]);
          if (lane == 0) S.part[warp * 6 + k] = v;
        }
      }
      __syncthreads();
      if (tid == 0) {
        float sumsd[6], dp[6];
        for (int k = 0; k < 6; ++k) {
          float s = S.part[k];
          if (!EX)
            for (int wv = 1; wv < nw; ++wv) s = s + S.part[wv * 6 + k];
          sumsd[k] = s;
        }
        lu6_solve(S.lu, sumsd, dp);                // 9b. odometer.cpp:407
        for (int k = 0; k < 6; ++k) S.p[k] += dp[k];   // 10. addpose_se3, pose.cpp:116-129
        se3_exp<float>(S.G, S.p);
        const float normdp = normdp_l1(dp);
        if (S.it == 0) S.normdp_init = normdp;
        S.normdp = normdp;
        if (trace && trace_n < prm.trace_cap)
          trace_record(trace + (int64_t)ICT_TRACE_FLOATS * trace_n++, sl, S.it, sumsd, dp, normdp, S.nvis);
        S.npix += (long long)S.nvis * n;
        S.nvis = 0;
        S.it += 1;
        S.cont = keep_iterating(op, S.it, S.normdp, S.normdp_init);
      }
      __syncthreads();
    }
    if (tid == 0) store_level_iters(prm.iters, op, t, sl, S.it);
  }

  if (tid == 0) finish_track(prm, t, donorm, S.p, S.G, prm.p_out, prm.npixres, S.npix, trace, trace_n);
}

// SetPose without TrackPose: pose.cpp:25-76 + project_pt at lv_l (what Get2DPoints returns, odometer.h:30)
__global__ void __launch_bounds__(128) k_reproject(const TrackParams prm) {
  __shared__ float s_p[6], s_G[12];
  const int t = blockIdx.x + prm.t0;
  const ict_optparam& op = prm.op;
  const int64_t off = prm.pt_off[t];
  const int n_in = (int)(prm.pt_off[t + 1] - off);
  const int P = min(n_in, op.maxpttrack);
  if (threadIdx.x == 0) track_setpose(prm.p_in, prm.norm, t, op.donorm != 0, s_p, s_G);
  __syncthreads();
  const float* q = prm.pt3d + 3 * off;
  for (int i = threadIdx.x; i < P; i += blockDim.x)
    save_rotated_point<false>(prm, s_G, off, n_in, i, q[i], q[n_in + i], q[2 * (int64_t)n_in + i], nullptr, nullptr, nullptr);
}

cudaError_t launch_reproject(const TrackParams& prm, cudaStream_t stream) {
  if (prm.T <= 0) return cudaSuccess;
  k_reproject<<<prm.T, 128, 0, stream>>>(prm);
  count_launch();
  return cudaGetLastError();
}


// ==================================================================================================
// K2f — the production form of K2 for the default settings (tree reductions, no patch normalisation,
// psz in {8,16,32}).  Same arithmetic per pixel and per track as k_track above (which stays as the
// general path: any psz, dopatchnorm, reference-order sums); what changes is the work decomposition:
//
//  * a warp owns a contiguous run of "groups" (32*KT pixels of one point; for psz 32: four consecutive
//    patch rows, lane = column), so everything that is constant per point — the ten SD coefficients,
//    the bilinear weights, the patch origin, the visibility — sits in registers and is recomputed only
//    when the warp moves to another point; no per-point shared-memory traffic in the pixel loop;
//  * every warp projects the points it works on itself (a dozen flops, all lanes redundantly), so the
//    iteration needs two CTA barriers instead of three and no per-point staging arrays;
//  * for psz 32 the row above is carried in registers from one row to the next: 10 gathers per 4
//    pixels instead of 16 (30 instead of 48 in the template precompute);
//  * template gather and Hessian accumulation are one pass;
//  * the cross-warp sums are done by six (21) lanes of warp 0 in parallel before lane 0 solves.
// Shared memory per CTA: 12 B per template pixel + 64 B per point; four CTAs per SM.
// ==================================================================================================
struct FastShared {
  float G[12];
  float p[6];
  float sum[8];
  float dp[6];
  float part[8 * 24];
  float Hsum[21];
  Lu6 lu;
  float normdp, normdp_init, lvl_cycles;
  int cont, it;
  long long npix;
};

template <int PSZ, int KTMAX, int MINB>
__global__ void __launch_bounds__(256, MINB) k_track_fast(const TrackParams prm) {
  constexpr int N = PSZ * PSZ;                      // pixels per patch
  constexpr int KT = (N / 32 < KTMAX) ? N / 32 : KTMAX;   // 32-pixel steps per group
  constexpr int GE = 32 * KT;                       // pixels per group
  constexpr int GPP = N / GE;                       // groups per point
  extern __shared__ __align__(16) float smem[];
  __shared__ FastShared S;

  const int t = blockIdx.x + prm.t0;
  const ict_optparam& op = prm.op;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
  const int pszd2 = PSZ / 2;
  const int64_t off = prm.pt_off[t];
  const int n_in = (int)(prm.pt_off[t + 1] - off);
  const int P = min(n_in, op.maxpttrack);
  const int E = P * N;
  const bool donorm = op.donorm != 0;

  float* s_ref = smem;
  float* s_gx = s_ref + E;
  float* s_gy = s_gx + E;
  float* s_X = s_gy + E;                            // per point: X Y Z (world) Xc Yc Zc (reference camera)
  float* s_Y = s_X + P;
  float* s_Z = s_Y + P;
  float* s_Xc = s_Z + P;
  float* s_Yc = s_Xc + P;
  float* s_Zc = s_Yc + P;
  float* s_coef = s_Zc + P;                         // [P][10], kept across levels for points that go out of view

  const TrackFrames fr = track_frames(prm, t);

  // this warp's run of groups
  const int G_all = P * GPP;
  const int gpw = (G_all + nw - 1) / nw;
  const int g_lo = min(warp * gpw, G_all), g_hi = min(g_lo + gpw, G_all);

  // ---- ResetOdometer + points ----------------------------------------------------------------------
  for (int e = tid; e < E; e += nt) { s_ref[e] = 0.0f; s_gx[e] = 0.0f; s_gy[e] = 0.0f; }
  {
    const float* q = prm.pt3d + 3 * off;
    for (int i = tid; i < P; i += nt) {
      s_X[i] = q[i];
      s_Y[i] = q[n_in + i];
      s_Z[i] = q[2 * (int64_t)n_in + i];
#pragma unroll
      for (int k = 0; k < 10; ++k) s_coef[i * 10 + k] = 0.0f;
    }
  }
  if (tid == 0) {
    track_setpose_from(prm, prm.p_in, t, donorm, S.p, S.G, S.Hsum);
    S.npix = 0;
  }
  __syncthreads();
  for (int i = tid; i < P; i += nt) save_rotated_point(prm, S.Hsum, off, n_in, i, s_X[i], s_Y[i], s_Z[i], s_Xc, s_Yc, s_Zc);
  __syncthreads();

  float* trace = track_trace(prm, t);
  int trace_n = 0;

  for (int sl = op.lv_f; sl >= op.lv_l; --sl) {
    const float fx = prm.cam.fx[sl], fy = prm.cam.fy[sl], cx = prm.cam.cx[sl], cy = prm.cam.cy[sl];
    const float swo = prm.cam.swo[sl], sho = prm.cam.sho[sl];
    const int width = prm.cam.width[sl];
    const float* __restrict__ Iref = fr.ref->I[sl];
    const float* __restrict__ Dxr = fr.ref->dx[sl];
    const float* __restrict__ Dyr = fr.ref->dy[sl];
    const float* __restrict__ Inew = fr.nw->I[sl];

    // ---- 4+5+6: template gather, SD coefficients, Hessian — one pass over this warp's groups ------------
    {
      float acc[21];
#pragma unroll
      for (int k = 0; k < 21; ++k) acc[k] = 0.0f;
      int cur = -1;
      bool vis = false;
      PatchPlace pl = {0, 0.f, 0.f, 0.f, 0.f};
      float cf[10];
#pragma unroll
      for (int k = 0; k < 10; ++k) cf[k] = 0.0f;
      float sxx = 0.0f, sxy = 0.0f, syy = 0.0f;     // sums of dx*dx, dx*dy, dy*dy of the current point
      for (int g = g_lo; g < g_hi; ++g) {
        const int i = g / GPP, gp = g - i * GPP;
        if (i != cur) {
          fold_hessian(acc, cf, sxx, sxy, syy);
          sxx = sxy = syy = 0.0f;
          cur = i;
          const float xc = s_Xc[i], yc = s_Yc[i], zc = s_Zc[i];
          const float mx = (xc / zc) * fx + cx, my = (yc / zc) * fy + cy;
          vis = (mx >= 0) & (my >= 0) & (mx <= swo) & (my <= sho);      // odometer.cpp:273-275
          if (vis) {
            pl = patch_place(mx, my, pszd2, width);
            sd_coefs(xc, yc, zc, fx, fy, cf);
            if (gp == 0) {                                                // persists for later levels
#pragma unroll
              for (int k = 0; k < 10; ++k)
                if (lane == k) s_coef[i * 10 + k] = cf[k];
            }
          } else {
#pragma unroll
            for (int k = 0; k < 10; ++k) cf[k] = s_coef[i * 10 + k];      // stale coefficients (SURVEY §9.6)
          }
        }
        const int ebase = i * N + gp * GE + lane;
        if (vis) {
          if (PSZ == 32) {
            const int a0 = pl.base + (gp * KT) * width + lane;
            float ci = __ldg(Iref + a0 - width), di = __ldg(Iref + a0 - width - 1);
            float cx_ = __ldg(Dxr + a0 - width), dx_ = __ldg(Dxr + a0 - width - 1);
            float cy_ = __ldg(Dyr + a0 - width), dy_ = __ldg(Dyr + a0 - width - 1);
#pragma unroll
            for (int j = 0; j < KT; ++j) {
              const int a = a0 + j * width;
              const float ai = __ldg(Iref + a), bi = __ldg(Iref + a - 1);
              const float ax = __ldg(Dxr + a), bx = __ldg(Dxr + a - 1);
              const float ay = __ldg(Dyr + a), by = __ldg(Dyr + a - 1);
              s_ref[ebase + 32 * j] = ((pl.w0 * ai + pl.w1 * bi) + pl.w2 * ci) + pl.w3 * di;
              s_gx[ebase + 32 * j] = ((pl.w0 * ax + pl.w1 * bx) + pl.w2 * cx_) + pl.w3 * dx_;
              s_gy[ebase + 32 * j] = ((pl.w0 * ay + pl.w1 * by) + pl.w2 * cy_) + pl.w3 * dy_;
              ci = ai; di = bi; cx_ = ax; dx_ = bx; cy_ = ay; dy_ = by;
            }
          } else {
#pragma unroll
            for (int j = 0; j < KT; ++j) {
              const int q = gp * GE + 32 * j + lane, r = q / PSZ, c = q - r * PSZ;
              const int a = pl.base + r * width + c;
              s_ref[ebase + 32 * j] = bilin4(Iref, a, width, pl.w0, pl.w1, pl.w2, pl.w3);
              s_gx[ebase + 32 * j] = bilin4(Dxr, a, width, pl.w0, pl.w1, pl.w2, pl.w3);
              s_gy[ebase + 32 * j] = bilin4(Dyr, a, width, pl.w0, pl.w1, pl.w2, pl.w3);
            }
          }
        }
#pragma unroll
        for (int j = 0; j < KT; ++j) {   // own writes: no barrier needed
          const float gx = s_gx[ebase + 32 * j], gy = s_gy[ebase + 32 * j];
          sxx = sxx + gx * gx;
          sxy = sxy + gx * gy;
          syy = syy + gy * gy;
        }
      }
      fold_hessian(acc, cf, sxx, sxy, syy);
      warp_sum_store<21>(acc, &S.part[warp * 24]);
    }
    __syncthreads();
    if (warp == 0) {                                // the serial sections: Hessian sums + LU, solve + update
      const long long t_lv0 = trace ? clock64() : 0;
      if (lane < 21) {
        float v[8];
#pragma unroll
        for (int wv = 0; wv < 8; ++wv) v[wv] = wv < nw ? S.part[wv * 24 + lane] : 0.0f;
        float s = v[0];
#pragma unroll
        for (int wv = 1; wv < 8; ++wv) s = wv < nw ? s + v[wv] : s;
        S.Hsum[lane] = s;
      }
      __syncwarp();
      lu6_factor_warp(S.Hsum, S.lu);                // all 32 lanes; same elimination as Eigen's fullPivLu
      if (lane == 0) {
        S.normdp_init = 1e-10f;
        S.normdp = 1e-10f;
        S.it = 0;
        S.cont = keep_iterating(op, 0, 1e-10f, 1e-10f);
        S.lvl_cycles = (float)(clock64() - t_lv0);
      }
    }
    __syncthreads();

    // ---- iterations --------------------------------------------------------------------------------
    while (S.cont) {
      const long long t_it0 = trace ? clock64() : 0;   // instrumentation only (trace records [22], [23])
      float Gm[12];
#pragma unroll
      for (int k = 0; k < 12; ++k) Gm[k] = S.G[k];
      float acc[6];
#pragma unroll
      for (int k = 0; k < 6; ++k) acc[k] = 0.0f;
      int nvis = 0;   // points this warp is the first to touch and that are visible in the new frame
      int cur = -1;
      bool vis = false;
      PatchPlace pl = {0, 0.f, 0.f, 0.f, 0.f};
      float cf[10];
#pragma unroll
      for (int k = 0; k < 10; ++k) cf[k] = 0.0f;
      float ax = 0.0f, ay = 0.0f;                    // sums of dx*pdiff, dy*pdiff of the current point
      for (int g = g_lo; g < g_hi; ++g) {
        const int i = g / GPP, gp = g - i * GPP;
        if (i != cur) {
          fold_jtr(acc, cf, ax, ay);
          ax = ay = 0.0f;
          cur = i;
          float tx, ty, tz;                                     // project_pt, pose.cpp:307-397
          rigid_apply<float>(Gm, s_X[i], s_Y[i], s_Z[i], tx, ty, tz);
          const float mx = (tx / tz) * fx + cx, my = (ty / tz) * fy + cy;
          vis = (mx >= 0) & (my >= 0) & (mx <= swo) & (my <= sho);   // odometer.cpp:369-371
          if (vis) {
            pl = patch_place(mx, my, pszd2, width);
#pragma unroll
            for (int k = 0; k < 10; ++k) cf[k] = s_coef[i * 10 + k];
            nvis += (gp == 0);
          }
        }
        if (!vis) continue;
        const int ebase = i * N + gp * GE + lane;
        if (PSZ == 32) {
          const int a0 = pl.base + (gp * KT) * width + lane;
          float c_ = __ldg(Inew + a0 - width), d_ = __ldg(Inew + a0 - width - 1);
#pragma unroll
          for (int j = 0; j < KT; ++j) {
            const float a_ = __ldg(Inew + a0 + j * width), b_ = __ldg(Inew + a0 + j * width - 1);
            const float pn = ((pl.w0 * a_ + pl.w1 * b_) + pl.w2 * c_) + pl.w3 * d_;
            c_ = a_; d_ = b_;
            const float pd = s_ref[ebase + 32 * j] - pn;
            ax = ax + s_gx[ebase + 32 * j] * pd;
            ay = ay + s_gy[ebase + 32 * j] * pd;
          }
        } else {
#pragma unroll
          for (int j = 0; j < KT; ++j) {
            const int q = gp * GE + 32 * j + lane, r = q / PSZ, c = q - r * PSZ;
            const float pn = bilin4(Inew, pl.base + r * width + c, width, pl.w0, pl.w1, pl.w2, pl.w3);
            const float pd = s_ref[ebase + 32 * j] - pn;
            ax = ax + s_gx[ebase + 32 * j] * pd;
            ay = ay + s_gy[ebase + 32 * j] * pd;
          }
        }
      }
      fold_jtr(acc, cf, ax, ay);
      warp_sum6_store(acc, &S.part[warp * 24]);
      if (lane == 0) S.part[warp * 24 + 6] = (float)nvis;
      const long long t_par = trace ? clock64() : 0;
      __syncthreads();
      if (warp == 0) {
        const long long t_ser0 = trace ? clock64() : 0;
        if (lane < 7) {   // 9a. cross-warp sums, fixed order, seven lanes in parallel (loads issued together)
          float v[8];
#pragma unroll
          for (int wv = 0; wv < 8; ++wv) v[wv] = wv < nw ? S.part[wv * 24 + lane] : 0.0f;
          float s = v[0];
#pragma unroll
          for (int wv = 1; wv < 8; ++wv) s = wv < nw ? s + v[wv] : s;
          S.sum[lane] = s;
        }
        __syncwarp();
        const bool fullrank = S.lu.rank == 6;
        if (fullrank) {                              // 9b. odometer.cpp:407, six lanes + shuffles
          const float x = lu6_solve_warp_rcp(S.lu, S.sum);
          if (lane < 6) S.dp[lane] = x;
          __syncwarp();
        }
        if (lane == 0) {
          if (!fullrank) lu6_solve(S.lu, S.sum, S.dp);
          float dp[6], pr[6], Gr[12];                // registers: shared-memory operands would be re-read after every store
#pragma unroll
          for (int k = 0; k < 6; ++k) { dp[k] = S.dp[k]; pr[k] = S.p[k] + dp[k]; S.p[k] = pr[k]; }   // 10. addpose_se3
          Gr[3] = Gr[7] = Gr[11] = 0.0f;
          se3_exp_f32_series(Gr, pr);
#pragma unroll
          for (int k = 0; k < 12; ++k) S.G[k] = Gr[k];
          const float normdp = normdp_l1(dp);
          if (S.it == 0) S.normdp_init = normdp;
          S.normdp = normdp;
          const int nv = (int)S.sum[6];
          if (trace && trace_n < prm.trace_cap) {
            float* rec = trace + (int64_t)ICT_TRACE_FLOATS * trace_n++;
            trace_record(rec, sl, S.it, S.sum, dp, normdp, nv);
            rec[21] = S.lvl_cycles;                    // cycles of this level's Hessian sums + LU factorisation
            rec[22] = (float)(clock64() - t_ser0);     // cycles warp 0 spends in the serial section
            rec[23] = (float)(t_par - t_it0);          // cycles warp 0 spends in the parallel section
          }
          S.npix += (long long)nv * N;
          S.it += 1;
          S.cont = keep_iterating(op, S.it, S.normdp, S.normdp_init);
        }
      }
      __syncthreads();
    }
    if (tid == 0) store_level_iters(prm.iters, op, t, sl, S.it);
  }

  if (tid == 0) finish_track(prm, t, donorm, S.p, S.G, prm.p_out, prm.npixres, S.npix, trace, trace_n);
}

static size_t fast_smem_bytes(const ict_optparam& op, int max_pts) {
  const size_t P = (size_t)track_pcap(op, max_pts);
  return sizeof(float) * (3 * P * op.novals + 16 * P);
}

// Rows per group (KTMAX) x CTAs per SM (MINB) for psz 32, measured on one B200 (8 sequences), in pixel-residuals/s:
//   KT 4/4 CTAs 2.61e11   KT 4/3 CTAs 2.51e11   KT 8/4 2.75e11   KT 8/3 2.66e11   KT 16/4 2.80e11   KT 16/3 2.66e11
// More rows per group put more independent gathers in flight per warp, and four resident CTAs beat three even though
// 64 registers spill ~230 B in the per-level precompute.
size_t track_smem_bytes(const ict_optparam& op, int max_pts, int sum_mode) {
  const int P = track_pcap(op, max_pts);
  const size_t E = (size_t)P * op.novals;
  const size_t Epad = (E + 3) & ~(size_t)3;
  const size_t planes = (op.dopatchnorm || sum_mode) ? 4 : 3;
  return sizeof(float) * (planes * Epad + (size_t)23 * P) + 16;
}

// the general kernel sets no carve-out
template <int PSZ>
static cudaError_t launch_track_p(const TrackParams& prm, size_t smem, int nt, int mode, cudaStream_t stream) {
  switch (mode) {
    case 0: return launch_cta_kernel<k_track<PSZ, 0>>(prm.T, nt, smem, -1, stream, prm);
    case 1: return launch_cta_kernel<k_track<PSZ, 1>>(prm.T, nt, smem, -1, stream, prm);
    case 2: return launch_cta_kernel<k_track<PSZ, 2>>(prm.T, nt, smem, -1, stream, prm);
    case 3: return launch_cta_kernel<k_track<PSZ, 3>>(prm.T, nt, smem, -1, stream, prm);
    case 6: return launch_cta_kernel<k_track<PSZ, 6>>(prm.T, nt, smem, -1, stream, prm);
    default: return launch_cta_kernel<k_track<PSZ, 7>>(prm.T, nt, smem, -1, stream, prm);
  }
}

TrackKernel select_track_kernel(const ict_optparam& op, int max_pts, int sum_mode, int eigen_packet, int force_general,
                                int no_k2r, int tma_ok) {
  const bool general_fits = track_smem_bytes(op, max_pts, sum_mode) <= (size_t)ICT_TRACK_SMEM_LIMIT;
  if (!force_general && sum_mode == 0) {
    if (v8_supported(op, max_pts)) return TrackKernel::V8;           // 8x8 patches, with or without dopatchnorm
    if (general_fits && !op.dopatchnorm) {
      if (op.psz == 32 && v2_smem_bytes(op, max_pts) <= (size_t)ICT_TRACK_SMEM_LIMIT) return TrackKernel::V2;
      if (op.psz == 8 || op.psz == 16 || op.psz == 32) return TrackKernel::Fast;
    }
  }
  if (!force_general && sum_mode != 0) {
    if (kx8_supported(op, max_pts)) return TrackKernel::X8;          // 8x8 (+/- dopatchnorm) and 16x16 patches
    // K2r and K2x run the eight chains of 4-float packets only: with 8-float packets psz 32 takes the general kernel
    if (general_fits && !op.dopatchnorm && eigen_packet == 4) {
      if (!no_k2r && kr_supported(op, max_pts, tma_ok)) return TrackKernel::R;
      if (op.psz == 32 && kx_smem_bytes(op, max_pts) <= (size_t)ICT_TRACK_SMEM_LIMIT) return TrackKernel::X;
    }
  }
  return general_fits ? TrackKernel::General : TrackKernel::MultiCta;
}

cudaError_t launch_track(const TrackParams& prm, TrackKernel k, int max_pts, cudaStream_t stream) {
  if (prm.T <= 0) return cudaSuccess;
  if (prm.seq_n > 1 && k != TrackKernel::V8) return cudaErrorInvalidConfiguration;   // only K2v8 loops over frames
  if (prm.seq_n > 1 && prm.p_start) return cudaErrorInvalidConfiguration;         // a chain starts each step at p_in
  const int P = track_pcap(prm.op, max_pts);
  const long long E = (long long)P * prm.op.novals;
  const int nt = E >= 2048 ? 256 : (E >= 512 ? 128 : 64);
  switch (k) {
    case TrackKernel::V8: return launch_track_v8(prm, max_pts, stream);
    case TrackKernel::V2: return launch_track_v2(prm, max_pts, stream);
    case TrackKernel::Fast: {
      const size_t smem = fast_smem_bytes(prm.op, max_pts);
      switch (prm.op.psz) {
        case 8: return launch_cta_kernel<k_track_fast<8, 4, 4>>(prm.T, nt, smem, 100, stream, prm);
        case 16: return launch_cta_kernel<k_track_fast<16, 4, 4>>(prm.T, nt, smem, 100, stream, prm);
        default: return launch_cta_kernel<k_track_fast<32, 16, 4>>(prm.T, nt, smem, 100, stream, prm);
      }
    }
    case TrackKernel::X8: return launch_track_x8(prm, max_pts, stream);
    case TrackKernel::R: return launch_track_r(prm, max_pts, stream);
    case TrackKernel::X: return launch_track_x(prm, max_pts, stream);
    case TrackKernel::General: {
      const size_t smem = track_smem_bytes(prm.op, max_pts, prm.sum_mode);
      const int mode = (prm.op.dopatchnorm ? 1 : 0) | (prm.sum_mode ? 2 : 0) | (prm.sum_mode && prm.eigen_packet == 8 ? 4 : 0);
      const int ntx = (mode & 2) && nt < 192 ? 192 : nt;   // the reference-order J^T r needs 6*16 = 96 threads, the Hessian
                                                           // 21*8 = 168 (it loops over the 21*16 chains of 8-float packets)
      switch (prm.op.psz) {
        case 8: return launch_track_p<8>(prm, smem, ntx, mode, stream);
        case 16: return launch_track_p<16>(prm, smem, ntx, mode, stream);
        case 32: return launch_track_p<32>(prm, smem, ntx, mode, stream);
        default: return launch_track_p<0>(prm, smem, ntx, mode, stream);
      }
    }
    default: return cudaErrorInvalidConfiguration;   // MultiCta: launch_track_big, one track at a time
  }
}

}  // namespace ict
