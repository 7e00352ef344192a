// ict_patches.cu — patch extraction (util_getPatch / util_getPatch_grad for a list of centres) and the NCC hypothesis
// scoring kernel.
#include "ict_kernels.cuh"
#include "ict_device.cuh"

namespace ict {

// ==================================================================================================
// util_getPatch / util_getPatch_grad (utilities.cpp:55-113, 115-189) for a list of patch centres: one CTA per centre,
// bilinear samples with the reference's placement (ceil(x + 1e-5f) quirk included) and association order, optional
// mean subtraction of the INTENSITY patch with Eigen's packet sum (utilities.cpp:111-112, 187-188).
// planes: bit 0 intensity, bit 1 dx, bit 2 dy.  out_* : [npatch][psz*psz].
// ==================================================================================================
__global__ void __launch_bounds__(128) k_get_patches(const float* __restrict__ I, const float* __restrict__ dx,
                                                     const float* __restrict__ dy, int width, int psz, int pszd2,
                                                     int patchnorm, const float* __restrict__ mids, float* out_I,
                                                     float* out_dx, float* out_dy) {
  const int n = psz * psz;
  const long long g = blockIdx.x;
  const float mx = mids[2 * g], my = mids[2 * g + 1];
  const PatchPlace q = patch_place(mx, my, pszd2, width);
  for (int e = threadIdx.x; e < n; e += blockDim.x) {
    const int r = e / psz, c = e - r * psz, ad = q.base + r * width + c;
    if (out_I) out_I[g * n + e] = bilin4(I, ad, width, q.w0, q.w1, q.w2, q.w3);
    if (out_dx) out_dx[g * n + e] = bilin4(dx, ad, width, q.w0, q.w1, q.w2, q.w3);
    if (out_dy) out_dy[g * n + e] = bilin4(dy, ad, width, q.w0, q.w1, q.w2, q.w3);
  }
  if (patchnorm && out_I) {
    __shared__ float s_mean;
    __syncthreads();
    if (threadIdx.x == 0) {
      float* p = out_I + g * n;
      s_mean = eigen_sum_serial<4>([&](int e) { return p[e]; }, n) / n;   // tmp_in_e.sum() / novals
    }
    __syncthreads();
    for (int e = threadIdx.x; e < n; e += blockDim.x) out_I[g * n + e] = out_I[g * n + e] - s_mean;
  }
}

cudaError_t launch_get_patches(const float* I, const float* dx, const float* dy, int width, int psz, int pszd2,
                               int patchnorm, int npatch, const float* mids, float* out_I, float* out_dx, float* out_dy,
                               cudaStream_t stream) {
  if (npatch <= 0) return cudaSuccess;
  k_get_patches<<<npatch, 128, 0, stream>>>(I, dx, dy, width, psz, pszd2, patchnorm, mids, out_I, out_dx, out_dy);
  count_launch();
  return cudaGetLastError();
}

// ==================================================================================================
// NCC hypothesis scoring, run_track_nposes.cpp:271-355.  One CTA per point; three mean-subtracted psz x psz
// patches (util_getPatch with dopatchnorm, :281) at level lv_l, each divided by its norm (:317-319),
// corr = max(0, (max(0,<b,r>)*nback^2 + max(0,<r,f>)*nfwd^2) / (nback^2 + nfwd^2)) (:324-348).
// Stale patches of invalid points never reach the output in the reference (their weight is 0), so points are
// independent.
// ==================================================================================================
__device__ __forceinline__ float cta_sum(float v, float* s_red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) s_red[warp] = v;
  __syncthreads();
  float s = s_red[0];
  for (int wv = 1; wv < nw; ++wv) s = s + s_red[wv];
  return s;
}

__global__ void __launch_bounds__(128) k_ncc(ict_optparam op, CamLevels cam, const float* __restrict__ img_b,
                                             const float* __restrict__ img_r, const float* __restrict__ img_f,
                                             int nback, int nfwd, const int64_t* __restrict__ pt_off, int T,
                                             const float* __restrict__ pb, const float* __restrict__ pr,
                                             const float* __restrict__ pf, float* __restrict__ out) {
  extern __shared__ float sm[];
  __shared__ float s_red[4];
  __shared__ int s_t;
  const int n = op.novals, psz = op.psz, l = op.lv_l;
  const long long g = blockIdx.x;   // global point index
  if (threadIdx.x == 0) {
    int lo = 0, hi = T;             // track with pt_off[t] <= g < pt_off[t+1]
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (pt_off[mid] <= g) lo = mid; else hi = mid; }
    s_t = lo;
  }
  __syncthreads();
  const int t = s_t;
  const int64_t off = pt_off[t];
  const int n_t = (int)(pt_off[t + 1] - off);
  const int i = (int)(g - off);
  const float swo = cam.swo[l], sho = cam.sho[l];
  const int width = cam.width[l];
  const float* imgs[3] = {img_b, img_r, img_f};
  const float* pts[3] = {pb, pr, pf};
  bool val[3];
  float nrm[3];
  for (int k = 0; k < 3; ++k) {
    float* buf = sm + k * n;
    const float mx = pts[k][2 * off + i], my = pts[k][2 * off + n_t + i];
    val[k] = (mx > 0) & (my > 0) & (mx < swo) & (my < sho);   // strict, :292,299,307
    float ss = 0.0f;
    if (val[k]) {
      const PatchPlace q = patch_place(mx, my, op.pszd2, width);
      float s = 0.0f;
      for (int e = threadIdx.x; e < n; e += blockDim.x) {
        const int r = e / psz, c = e - r * psz;
        const float v = bilin4(imgs[k], q.base + r * width + c, width, q.w0, q.w1, q.w2, q.w3);
        buf[e] = v;
        s = s + v;
      }
      const float m = cta_sum(s, s_red) / n;
      for (int e = threadIdx.x; e < n; e += blockDim.x) {
        const float v = buf[e] - m;
        buf[e] = v;
        ss = ss + v * v;
      }
    } else {
      for (int e = threadIdx.x; e < n; e += blockDim.x) buf[e] = 0.0f;
    }
    nrm[k] = sqrtf(cta_sum(ss, s_red));
  }
  float corr = -1.0f;
  if (val[1]) {
    float d0 = 0.0f, d1 = 0.0f;
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
      const float b = sm[e] / nrm[0], r = sm[n + e] / nrm[1], f = sm[2 * n + e] / nrm[2];
      d0 = d0 + b * r;
      d1 = d1 + r * f;
    }
    d0 = cta_sum(d0, s_red);
    d1 = cta_sum(d1, s_red);
    float corr_br, corr_rf, w0, w1;
    if (val[0]) { corr_br = 0.0f < d0 ? d0 : 0.0f; w0 = (float)(nback * nback); } else { corr_br = -1.0f; w0 = 0.0f; }
    if (val[2]) { corr_rf = 0.0f < d1 ? d1 : 0.0f; w1 = (float)(nfwd * nfwd); } else { corr_rf = -1.0f; w1 = 0.0f; }
    const float v = (corr_br * w0 + corr_rf * w1) / (w0 + w1);
    corr = 0.0f < v ? v : 0.0f;
  }
  if (threadIdx.x == 0) out[g] = corr;
}

cudaError_t launch_ncc(const ict_optparam& op, const CamLevels& cam, const float* img_b, const float* img_r,
                       const float* img_f, int nback, int nfwd, const int64_t* pt_off, int T, const float* pb,
                       const float* pr, const float* pf, float* out, cudaStream_t stream) {
  // total points = pt_off[T] lives on the device; the caller passes host-known totals through T tracks
  int64_t total = 0;
  cudaError_t e = cudaMemcpyAsync(&total, pt_off + T, sizeof(int64_t), cudaMemcpyDeviceToHost, stream);
  if (e != cudaSuccess) return e;
  e = cudaStreamSynchronize(stream);
  if (e != cudaSuccess) return e;
  if (total <= 0) return cudaSuccess;
  const size_t smem = sizeof(float) * 3 * (size_t)op.novals;
  if (smem > 200 * 1024) return cudaErrorInvalidConfiguration;
  e = set_kernel_attrs<k_ncc>(200 * 1024, -1);
  if (e != cudaSuccess) return e;
  k_ncc<<<(unsigned)total, 128, smem, stream>>>(op, cam, img_b, img_r, img_f, nback, nfwd, pt_off, T, pb, pr, pf, out);
  count_launch();
  return cudaGetLastError();
}

}  // namespace ict
