// ict_evaluate.cu — ict_track_evaluate: one Gauss-Newton measurement of every track at a pose the caller chooses.
// ict_track_evaluate_poses (second half of the file) measures K candidate poses per track against one template.
//
// For each track: the template state TrackPose holds when it reaches `level` (odometer.cpp:268-334, starting from the
// zeroed arrays of Set3Dpoints, stale slots included), one projection / new-frame patch / pdiff at p_cur
// (odometer.cpp:360-396), and the level's Hessian (ComputeHessian, :428-472), J^T r (:399-404), the fullPivLu step
// (:407), sum pdiff^2 and per-point sums of pdiff^2.  Nothing stays resident in one CTA, so tracks of any size work:
//
//   k_eval_pose      per track   setpose_se3 of p_ref and of p_cur
//   k_eval_points    per point   camera-frame point, the finest level in [level, lv_f] at which it is inside the
//                                reference image (its placement and steepest-descent coefficients), the placement
//                                at p_cur in the new frame, the visible-point count
//   k_eval_slots     per pixel   template gather at that level, sd_1..6 with the reference's roundings, new patch
//   k_eval_patch     per point   patch means (dopatchnorm), pdiff, the point's sum of pdiff^2
//   k_eval_chains    reference order: one thread per (track, quantity, chain) — Eigen's 2W sequential chains
//   k_eval_partials  tree order: one CTA per (track, 4096-pixel chunk), fixed-order partials
//   k_eval_solve     one warp per track: the 28 totals, lu6_factor_warp + lu6_solve, outputs
//
// The 28 quantities are the 21 Hessian entries (ComputeHessian's order), the 6 J^T r entries and sum pdiff^2.
// Compiled with -fmad=false like every unit of the library (ict_device.cuh).
#include "ict_device.cuh"
#include "ict_kernels.cuh"

#include <type_traits>

namespace ict {


#define ICT_EVAL_NQ 28          // 21 H + 6 J^T r + 1 SSR
#define ICT_EVAL_CHUNK 4096     // pixels per CTA of the tree-order partials

// flags of EvalPoint
#define EV_REF 1                // inside the reference image at some level of [level, lv_f]
#define EV_NEW 2                // inside the new image at p_cur
#define EV_KEPT 4               // one of the first maxpttrack points of its track

struct EvalPoint {
  float rw[4], nw[4];           // bilinear weights: reference (at level lvl), new frame
  float coef[10];               // sd_coefs at lvl
  int rbase, nbase, lvl, flags, track, pad;
};

// ComputeHessian's pairs (a, b), a <= b, in its order (odometer.cpp:430-455)
__constant__ unsigned char c_qa[21] = {0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 4, 4, 5};
__constant__ unsigned char c_qb[21] = {0, 1, 2, 3, 4, 5, 1, 2, 3, 4, 5, 2, 3, 4, 5, 3, 4, 5, 4, 5, 5};

// the value quantity q contributes at pixel slot s (products rounded to fp32 per element, as Eigen's (x*y).sum())
__device__ __forceinline__ float eval_value(const EvalArgs& a, int q, int64_t s) {
  if (q < 21) return a.sd[c_qa[q] * a.S + s] * a.sd[c_qb[q] * a.S + s];
  if (q < 27) return a.sd[(q - 21) * a.S + s] * a.pd[s];
  return a.pd[s] * a.pd[s];
}

// track of a global index: the last t with off[t] <= g (off non-decreasing, off[0] = 0)
__device__ __forceinline__ int eval_track_of(const int64_t* off, int T, int64_t g) {
  int lo = 0, hi = T - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (off[mid] <= g) lo = mid; else hi = mid - 1;
  }
  return lo;
}

__global__ void __launch_bounds__(128) k_eval_pose(const EvalArgs a) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= a.T) return;
  const double* nm = a.norm + 4 * (int64_t)t;
  float p[6], G[12];
  setpose_se3(a.p_ref + 6 * (int64_t)t, a.op.donorm != 0, nm, nm[3], p, G);
  for (int k = 0; k < 12; ++k) a.G_ref[12 * (int64_t)t + k] = G[k];
  setpose_se3((a.p_cur ? a.p_cur : a.p_ref) + 6 * (int64_t)t, a.op.donorm != 0, nm, nm[3], p, G);
  for (int k = 0; k < 12; ++k) a.G_cur[12 * (int64_t)t + k] = G[k];
}

__global__ void __launch_bounds__(256) k_eval_points(const EvalArgs a) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= a.total) return;
  const int t = eval_track_of(a.pt_off, a.T, g);
  const int64_t off = a.pt_off[t];
  const int n_in = (int)(a.pt_off[t + 1] - off);
  const int i = (int)(g - off);
  EvalPoint q;
  for (int k = 0; k < 4; ++k) q.rw[k] = q.nw[k] = 0.0f;
  for (int k = 0; k < 10; ++k) q.coef[k] = 0.0f;
  q.rbase = q.nbase = 0;
  q.lvl = -1;
  q.flags = 0;
  q.track = t;
  q.pad = 0;
  if (i < a.op.maxpttrack) {
    q.flags = EV_KEPT;
    const float* pts = a.pt3d + 3 * off;
    const float X = pts[i], Y = pts[n_in + i], Z = pts[2 * (int64_t)n_in + i];
    const float* G = a.G_ref + 12 * (int64_t)t;
    // project_pt_save_rotated at the SetPose pose (pose.cpp:400-488)
    const float xc = G[0] * X + G[1] * Y + G[2] * Z + G[3];
    const float yc = G[4] * X + G[5] * Y + G[6] * Z + G[7];
    const float zc = G[8] * X + G[9] * Y + G[10] * Z + G[11];
    // TrackPose overwrites a point's template slots at every level where it is inside the reference image
    // (odometer.cpp:273-275) and leaves them otherwise: at `level` they hold the finest such level's
    float mx = 0.0f, my = 0.0f;
    for (int sl = a.op.lv_f; sl >= a.level; --sl) {
      const float x = (xc / zc) * a.cam.fx[sl] + a.cam.cx[sl];
      const float y = (yc / zc) * a.cam.fy[sl] + a.cam.cy[sl];
      if ((x >= 0) & (y >= 0) & (x <= a.cam.swo[sl]) & (y <= a.cam.sho[sl])) { q.lvl = sl; mx = x; my = y; }
    }
    if (q.lvl >= 0) {
      q.flags |= EV_REF;
      const PatchPlace pl = patch_place(mx, my, a.op.pszd2, a.cam.width[q.lvl]);
      q.rbase = pl.base;
      q.rw[0] = pl.w0; q.rw[1] = pl.w1; q.rw[2] = pl.w2; q.rw[3] = pl.w3;
      sd_coefs(xc, yc, zc, a.cam.fx[q.lvl], a.cam.fy[q.lvl], q.coef);
    }
    // project_pt at p_cur + the new-frame test (odometer.cpp:360-371)
    const float* H = a.G_cur + 12 * (int64_t)t;
    const float tx = H[0] * X + H[1] * Y + H[2] * Z + H[3];
    const float ty = H[4] * X + H[5] * Y + H[6] * Z + H[7];
    const float tz = H[8] * X + H[9] * Y + H[10] * Z + H[11];
    const int l = a.level;
    const float nx = (tx / tz) * a.cam.fx[l] + a.cam.cx[l];
    const float ny = (ty / tz) * a.cam.fy[l] + a.cam.cy[l];
    if ((nx >= 0) & (ny >= 0) & (nx <= a.cam.swo[l]) & (ny <= a.cam.sho[l])) {
      q.flags |= EV_NEW;
      const PatchPlace pl = patch_place(nx, ny, a.op.pszd2, a.cam.width[l]);
      q.nbase = pl.base;
      q.nw[0] = pl.w0; q.nw[1] = pl.w1; q.nw[2] = pl.w2; q.nw[3] = pl.w3;
      atomicAdd(a.nvis + t, 1);
    }
  }
  a.pts[g] = q;
}

__global__ void __launch_bounds__(256) k_eval_slots(const EvalArgs a) {
  const int n = a.op.novals;
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= a.S) return;
  const int64_t g = s / n;
  const int k = (int)(s - g * n), r = k / a.op.psz, c = k - r * a.op.psz;
  const EvalPoint& q = a.pts[g];
  float ref = 0.0f, pn = 0.0f, sd[6] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
  if (q.flags & EV_REF) {   // util_getPatch_grad at the point's level (utilities.cpp:115-189), sd as odometer.cpp:317-326
    const FrameDesc& fr = a.frames[a.ref_frame[q.track]];
    const int w = a.cam.width[q.lvl], addr = q.rbase + r * w + c;
    ref = bilin4(fr.I[q.lvl], addr, w, q.rw[0], q.rw[1], q.rw[2], q.rw[3]);
    const float gx = bilin4(fr.dx[q.lvl], addr, w, q.rw[0], q.rw[1], q.rw[2], q.rw[3]);
    const float gy = bilin4(fr.dy[q.lvl], addr, w, q.rw[0], q.rw[1], q.rw[2], q.rw[3]);
    sd_values(gx, gy, q.coef, sd);
  }
  if (q.flags & EV_NEW) {   // util_getPatch (utilities.cpp:55-113), mean subtracted later
    const int w = a.cam.width[a.level];
    pn = bilin4(a.frames[a.new_frame[q.track]].I[a.level], q.nbase + r * w + c, w, q.nw[0], q.nw[1], q.nw[2], q.nw[3]);
  }
  for (int j = 0; j < 6; ++j) a.sd[j * a.S + s] = sd[j];
  a.ref[s] = ref;
  a.pd[s] = pn;
}

// per point: patch means in Eigen's packet order (utilities.cpp:111-112, 187-188), pdiff (odometer.cpp:381), the
// point's sum of pdiff^2 in the same order
template <int W>
__global__ void __launch_bounds__(128) k_eval_patch(const EvalArgs a) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= a.total) return;
  const int n = a.op.novals;
  const int flags = a.pts[g].flags;
  float* ref = a.ref + g * n;
  float* pd = a.pd + g * n;
  if (!(flags & EV_NEW)) {
    for (int k = 0; k < n; ++k) pd[k] = 0.0f;
    if (a.pt_ssr) a.pt_ssr[g] = -1.0f;
    return;
  }
  const bool pn = a.op.dopatchnorm != 0;
  const float mref = (pn && (flags & EV_REF)) ? eigen_sum_serial<W>([&](int e) { return ref[e]; }, n) / n : 0.0f;
  const float mnew = pn ? eigen_sum_serial<W>([&](int e) { return pd[e]; }, n) / n : 0.0f;
  for (int k = 0; k < n; ++k) pd[k] = (ref[k] - mref) - (pd[k] - mnew);
  if (a.pt_ssr) a.pt_ssr[g] = eigen_sum_serial<W>([&](int e) { return pd[e] * pd[e]; }, n);
}

// reference order: chain c of quantity q of track t, thread (t * 28 + q) * 2W + c
template <int W>
__global__ void __launch_bounds__(256) k_eval_chains(const EvalArgs a) {
  constexpr int NCH = 2 * W;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)a.T * ICT_EVAL_NQ * NCH) return;
  const int c = (int)(idx % NCH), q = (int)((idx / NCH) % ICT_EVAL_NQ), t = (int)(idx / (NCH * ICT_EVAL_NQ));
  const int n = a.op.novals;
  const int64_t base = a.pt_off[t] * n;
  const int P = min((int)(a.pt_off[t + 1] - a.pt_off[t]), a.op.maxpttrack);
  const int N = a.op.maxpttrack * n, E = P * n;
  // eigen_chain<W>(v, c, as2, E) with the values of eight steps loaded ahead of their (still sequential) additions: the
  // same sum, but a long chain (dense tracks) is no longer one dependent global load per addition
  auto v = [&](int e) { return eval_value(a, q, base + e); };
  const int as2 = (N / NCH) * NCH;
  if (c >= as2) { a.chains[idx] = 0.0f; return; }
  float s = c < E ? v(c) : 0.0f;
  const int lim = as2 < E ? as2 : E;
  int e = c + NCH;
  for (; e + 7 * NCH < lim; e += 8 * NCH) {
    float x[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] = v(e + j * NCH);
#pragma unroll
    for (int j = 0; j < 8; ++j) s = s + x[j];
  }
  for (; e < lim; e += NCH) s = s + v(e);
  a.chains[idx] = s;
}

// tree order: CTA = one chunk of one track; per-thread strided sums, warp trees, warps in order
__global__ void __launch_bounds__(256) k_eval_partials(const EvalArgs a) {
  __shared__ float s_part[8][ICT_EVAL_NQ];
  const int chunk = blockIdx.x;
  const int t = eval_track_of(a.chunk_off, a.T, chunk);
  const int n = a.op.novals;
  const int64_t base = a.pt_off[t] * n;
  const int P = min((int)(a.pt_off[t + 1] - a.pt_off[t]), a.op.maxpttrack);
  const int E = P * n;
  const int e0 = (int)(chunk - a.chunk_off[t]) * ICT_EVAL_CHUNK, e1 = min(e0 + ICT_EVAL_CHUNK, E);
  float acc[ICT_EVAL_NQ];
#pragma unroll
  for (int k = 0; k < ICT_EVAL_NQ; ++k) acc[k] = 0.0f;
  for (int e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
    const int64_t s = base + e;
    float sd[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) sd[j] = a.sd[j * a.S + s];
    const float pd = a.pd[s];
    int k = 0;
#pragma unroll
    for (int x = 0; x < 6; ++x)
#pragma unroll
      for (int y = x; y < 6; ++y) { acc[k] = acc[k] + sd[x] * sd[y]; ++k; }
#pragma unroll
    for (int j = 0; j < 6; ++j) acc[21 + j] = acc[21 + j] + sd[j] * pd;
    acc[27] = acc[27] + pd * pd;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < ICT_EVAL_NQ; ++k) {
    const float v = warp_sum(acc[k]);
    if (lane == 0) s_part[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < ICT_EVAL_NQ) {
    float s = s_part[0][threadIdx.x];
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) s = s + s_part[w][threadIdx.x];
    a.partials[(int64_t)chunk * ICT_EVAL_NQ + threadIdx.x] = s;
  }
}

// one warp per track: totals, factor, solve, outputs
template <int W, bool REF>
__global__ void __launch_bounds__(128) k_eval_solve(const EvalArgs a) {
  __shared__ float s_sum[4][32];
  __shared__ Lu6 s_lu[4];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t = blockIdx.x * 4 + warp;
  if (t >= a.T) return;                 // whole warps leave together
  const int n = a.op.novals;
  const int64_t base = a.pt_off[t] * n;
  const int P = min((int)(a.pt_off[t + 1] - a.pt_off[t]), a.op.maxpttrack);
  const int N = a.op.maxpttrack * n, E = P * n;
  float v = 0.0f;
  if (lane < ICT_EVAL_NQ) {
    if (REF) {
      v = eigen_finish<W>(a.chains + ((int64_t)t * ICT_EVAL_NQ + lane) * (2 * W),
                          [&](int e) { return eval_value(a, lane, base + e); }, N, E);
    } else {
      for (int64_t c = a.chunk_off[t]; c < a.chunk_off[t + 1]; ++c) v = v + a.partials[c * ICT_EVAL_NQ + lane];
    }
  }
  s_sum[warp][lane] = v;
  __syncwarp();
  lu6_factor_warp(s_sum[warp], s_lu[warp]);
  if (a.lu && lane == 0) a.lu[t] = s_lu[warp];
  if (lane == 0) {
    float dp[6];
    lu6_solve(s_lu[warp], s_sum[warp] + 21, dp);
    if (a.out_dp)
      for (int k = 0; k < 6; ++k) a.out_dp[6 * (int64_t)t + k] = dp[k];
  }
  if (a.out_H && lane < 21) {
    const int x = c_qa[lane], y = c_qb[lane];
    a.out_H[36 * (int64_t)t + 6 * x + y] = v;
    a.out_H[36 * (int64_t)t + 6 * y + x] = v;
  }
  if (a.out_jtr && lane >= 21 && lane < 27) a.out_jtr[6 * (int64_t)t + lane - 21] = v;
  if (a.out_ssr && lane == 27) a.out_ssr[t] = v;
}

// ---- ict_track_evaluate_poses: K candidate poses per track against one template ------------------------------------
// The template, sd and H (with its factorisation) depend on p_ref only: they come from the kernels above, run once per
// track.  Per candidate only the new-image side is redone, with the sums in the order ict_track_evaluate uses, so the
// outputs for candidate k are its outputs at p_cur = candidate k bit for bit:
//
//   k_evp_template  per point              template - its mean (k_eval_patch's (ref - mref)), in place
//   k_evp_pose      per (track, candidate) setpose_se3 of the candidate
//   k_evp_points    per (point, candidate) placement at the candidate, the new-image test, visible count, patch mean
//   k_evp_chains    reference order: one thread per (track, chain, group of EVP_KG candidates), Eigen's 2W chains of
//                   the 6 J^T r sums and SSR; each template slot is read once for the group
//   k_evp_partials  tree order: one CTA per (chunk, group of EVP_KG candidates), k_eval_partials' tree per candidate
//   k_evp_solve     per (track, candidate): the 7 totals (eigen_finish or the chunks in order), lu6_solve with the
//                   track's factorisation
#define EVP_NQ 7                // 6 J^T r + 1 SSR
#define EVP_KG 4                // candidates per thread of the fused sums

struct EvalCand {
  float nw[4];                  // bilinear weights in the new frame
  int nbase, vis;               // patch origin, inside the new image
  float mnew;                   // new patch mean (dopatchnorm), else 0
  int pad;
};

template <int W>
__global__ void __launch_bounds__(128) k_evp_template(const EvalArgs a) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= a.total) return;
  const int n = a.op.novals;
  float* ref = a.ref + g * n;
  const bool pn = a.op.dopatchnorm != 0;
  const float mref = (pn && (a.pts[g].flags & EV_REF)) ? eigen_sum_serial<W>([&](int e) { return ref[e]; }, n) / n : 0.0f;
  for (int k = 0; k < n; ++k) ref[k] = ref[k] - mref;
}

__global__ void __launch_bounds__(128) k_evp_pose(const EvalArgs a, const EvalPoses b) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)a.T * b.K) return;
  const int t = (int)(idx / b.K);
  const double* nm = a.norm + 4 * (int64_t)t;
  float p[6], G[12];
  setpose_se3(b.p_cand + 6 * idx, a.op.donorm != 0, nm, nm[3], p, G);
  for (int k = 0; k < 12; ++k) b.G_cand[12 * idx + k] = G[k];
}

// k_eval_points' new-image half and k_eval_patch's mnew: point blockIdx.x * 256 + threadIdx.x at candidates
// blockIdx.y, blockIdx.y + gridDim.y, ...
template <int W>
__global__ void __launch_bounds__(256) k_evp_points(const EvalArgs a, const EvalPoses b) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= a.total) return;
  const int t = eval_track_of(a.pt_off, a.T, g);
  const int64_t off = a.pt_off[t];
  const int n_in = (int)(a.pt_off[t + 1] - off);
  const int i = (int)(g - off);
  const bool kept = i < a.op.maxpttrack;
  const float* pts = a.pt3d + 3 * off;
  const float X = kept ? pts[i] : 0.0f, Y = kept ? pts[n_in + i] : 0.0f, Z = kept ? pts[2 * (int64_t)n_in + i] : 0.0f;
  const int l = a.level;
  for (int k = blockIdx.y; k < b.K; k += gridDim.y) {
    EvalCand q;
    for (int j = 0; j < 4; ++j) q.nw[j] = 0.0f;
    q.nbase = q.vis = q.pad = 0;
    q.mnew = 0.0f;
    const float* H = b.G_cand + 12 * ((int64_t)t * b.K + k);
    const float tx = H[0] * X + H[1] * Y + H[2] * Z + H[3];
    const float ty = H[4] * X + H[5] * Y + H[6] * Z + H[7];
    const float tz = H[8] * X + H[9] * Y + H[10] * Z + H[11];
    const float nx = (tx / tz) * a.cam.fx[l] + a.cam.cx[l];
    const float ny = (ty / tz) * a.cam.fy[l] + a.cam.cy[l];
    if (kept && (nx >= 0) & (ny >= 0) & (nx <= a.cam.swo[l]) & (ny <= a.cam.sho[l])) {
      const PatchPlace pl = patch_place(nx, ny, a.op.pszd2, a.cam.width[l]);
      q.nbase = pl.base;
      q.nw[0] = pl.w0; q.nw[1] = pl.w1; q.nw[2] = pl.w2; q.nw[3] = pl.w3;
      q.vis = 1;
      atomicAdd(b.nvis + (int64_t)t * b.K + k, 1);
      if (a.op.dopatchnorm) {
        const int n = a.op.novals, psz = a.op.psz, w = a.cam.width[l], nb = pl.base;
        const float* img = a.frames[a.new_frame[t]].I[l];
        q.mnew = eigen_sum_serial<W>([=](int e) {
          const int r = e / psz;
          return bilin4(img, nb + r * w + (e - r * psz), w, pl.w0, pl.w1, pl.w2, pl.w3);
        }, n) / n;
      }
    }
    b.cand[g * b.K + k] = q;
  }
}

// pdiff of one slot at one candidate: k_eval_patch's (ref - mref) - (pn - mnew), 0 outside the new image
__device__ __forceinline__ float evp_pdiff(const EvalCand& q, const float* img, int w, int roff, float tref) {
  if (!q.vis) return 0.0f;
  const float pn = bilin4(img, q.nbase + roff, w, q.nw[0], q.nw[1], q.nw[2], q.nw[3]);
  return tref - (pn - q.mnew);
}

// acc[kk][0..6] (+)= the 7 values of track slot e (relative to the track's first slot) at candidates k0 .. k0+KG-1
// (those beyond K repeat candidate K-1 and are not stored)
template <bool FIRST>
__device__ __forceinline__ void evp_slot(const EvalArgs& a, const EvalPoses& b, const float* img, int64_t pt0, int e,
                                         int k0, float (&acc)[EVP_KG][EVP_NQ]) {
  const int n = a.op.novals, psz = a.op.psz, w = a.cam.width[a.level];
  const int i = e / n, pix = e - i * n, r = pix / psz, roff = r * w + (pix - r * psz);
  const int64_t g = pt0 + i, s = g * n + pix;
  float sd[6];
#pragma unroll
  for (int j = 0; j < 6; ++j) sd[j] = a.sd[j * a.S + s];
  const float tref = a.ref[s];
#pragma unroll
  for (int kk = 0; kk < EVP_KG; ++kk) {
    const float pd = evp_pdiff(b.cand[g * b.K + min(k0 + kk, b.K - 1)], img, w, roff, tref);
#pragma unroll
    for (int j = 0; j < 6; ++j) acc[kk][j] = FIRST ? sd[j] * pd : acc[kk][j] + sd[j] * pd;
    acc[kk][6] = FIRST ? pd * pd : acc[kk][6] + pd * pd;
  }
}

// reference order: chain c of candidates k0.. of track t; thread ((t * ngroups + group) * 2W + c)
template <int W>
__global__ void __launch_bounds__(256) k_evp_chains(const EvalArgs a, const EvalPoses b) {
  constexpr int NCH = 2 * W;
  const int ng = (b.K + EVP_KG - 1) / EVP_KG;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)a.T * ng * NCH) return;
  const int c = (int)(idx % NCH), k0 = (int)((idx / NCH) % ng) * EVP_KG, t = (int)(idx / ((int64_t)NCH * ng));
  const int n = a.op.novals;
  const int P = min((int)(a.pt_off[t + 1] - a.pt_off[t]), a.op.maxpttrack);
  const int N = a.op.maxpttrack * n, E = P * n;
  const int as2 = (N / NCH) * NCH;
  const float* img = a.frames[a.new_frame[t]].I[a.level];
  float acc[EVP_KG][EVP_NQ];
#pragma unroll
  for (int kk = 0; kk < EVP_KG; ++kk)
#pragma unroll
    for (int q = 0; q < EVP_NQ; ++q) acc[kk][q] = 0.0f;
  if (c < as2) {   // eigen_chain: the first value assigned, the rest added in sequence below min(as2, E)
    if (c < E) evp_slot<true>(a, b, img, a.pt_off[t], c, k0, acc);
    const int lim = as2 < E ? as2 : E;
    for (int e = c + NCH; e < lim; e += NCH) evp_slot<false>(a, b, img, a.pt_off[t], e, k0, acc);
  }
#pragma unroll
  for (int kk = 0; kk < EVP_KG; ++kk)
    if (k0 + kk < b.K)
#pragma unroll
      for (int q = 0; q < EVP_NQ; ++q) b.chains[(((int64_t)t * b.K + k0 + kk) * EVP_NQ + q) * NCH + c] = acc[kk][q];
}

// tree order: k_eval_partials' CTA (256 strided lanes, warp_sum, warps in order) for each of EVP_KG candidates
__global__ void __launch_bounds__(256) k_evp_partials(const EvalArgs a, const EvalPoses b) {
  __shared__ float s_part[8][EVP_KG * EVP_NQ];
  const int ng = (b.K + EVP_KG - 1) / EVP_KG;
  const int64_t chunk = blockIdx.x / ng;
  const int k0 = (int)(blockIdx.x - chunk * ng) * EVP_KG;
  const int t = eval_track_of(a.chunk_off, a.T, chunk);
  const int P = min((int)(a.pt_off[t + 1] - a.pt_off[t]), a.op.maxpttrack);
  const int E = P * a.op.novals;
  const int e0 = (int)(chunk - a.chunk_off[t]) * ICT_EVAL_CHUNK, e1 = min(e0 + ICT_EVAL_CHUNK, E);
  const float* img = a.frames[a.new_frame[t]].I[a.level];
  float acc[EVP_KG][EVP_NQ];
#pragma unroll
  for (int kk = 0; kk < EVP_KG; ++kk)
#pragma unroll
    for (int q = 0; q < EVP_NQ; ++q) acc[kk][q] = 0.0f;
  for (int e = e0 + threadIdx.x; e < e1; e += blockDim.x) evp_slot<false>(a, b, img, a.pt_off[t], e, k0, acc);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int kk = 0; kk < EVP_KG; ++kk)
#pragma unroll
    for (int q = 0; q < EVP_NQ; ++q) {
      const float v = warp_sum(acc[kk][q]);
      if (lane == 0) s_part[warp][kk * EVP_NQ + q] = v;
    }
  __syncthreads();
  if (threadIdx.x < EVP_KG * EVP_NQ && k0 + (int)threadIdx.x / EVP_NQ < b.K) {
    float s = s_part[0][threadIdx.x];
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) s = s + s_part[w][threadIdx.x];
    b.partials[(chunk * b.K + k0) * EVP_NQ + threadIdx.x] = s;
  }
}

// the value of quantity q (0..5 J^T r, 6 SSR) at track slot e and candidate k, for eigen_finish's odd packet and tail
__device__ __forceinline__ float evp_value(const EvalArgs& a, const EvalPoses& b, const float* img, int64_t pt0, int k,
                                           int q, int e) {
  const int n = a.op.novals, psz = a.op.psz, w = a.cam.width[a.level];
  const int i = e / n, pix = e - i * n, r = pix / psz;
  const int64_t g = pt0 + i, s = g * n + pix;
  const float pd = evp_pdiff(b.cand[g * b.K + k], img, w, r * w + (pix - r * psz), a.ref[s]);
  return q < 6 ? a.sd[q * a.S + s] * pd : pd * pd;
}

template <int W, bool REF>
__global__ void __launch_bounds__(128) k_evp_solve(const EvalArgs a, const EvalPoses b) {
  __shared__ float s_v[128][8];
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)a.T * b.K) return;
  const int t = (int)(idx / b.K), k = (int)(idx - (int64_t)t * b.K);
  float* v = s_v[threadIdx.x];
  if (REF) {
    const int n = a.op.novals;
    const int P = min((int)(a.pt_off[t + 1] - a.pt_off[t]), a.op.maxpttrack);
    const int N = a.op.maxpttrack * n, E = P * n;
    const float* img = a.frames[a.new_frame[t]].I[a.level];
    const int64_t pt0 = a.pt_off[t];
    for (int q = 0; q < EVP_NQ; ++q)
      v[q] = eigen_finish<W>(b.chains + (idx * EVP_NQ + q) * (2 * W),
                             [&](int e) { return evp_value(a, b, img, pt0, k, q, e); }, N, E);
  } else {
    for (int q = 0; q < EVP_NQ; ++q) {
      float s = 0.0f;
      for (int64_t c = a.chunk_off[t]; c < a.chunk_off[t + 1]; ++c) s = s + b.partials[(c * b.K + k) * EVP_NQ + q];
      v[q] = s;
    }
  }
  if (b.out_jtr)
    for (int j = 0; j < 6; ++j) b.out_jtr[6 * idx + j] = v[j];
  if (b.out_ssr) b.out_ssr[idx] = v[6];
  if (b.out_dp) {
    float dp[6];
    lu6_solve(a.lu[t], v, dp);
    for (int j = 0; j < 6; ++j) b.out_dp[6 * idx + j] = dp[j];
  }
}

size_t evaluate_workspace(EvalArgs& a, int64_t nchunks, void* base) {
  size_t off = 0;
  auto take = [&](auto*& p, int64_t count) {
    using E = std::remove_reference_t<decltype(*p)>;
    off = (off + 255) & ~(size_t)255;
    if (base) p = reinterpret_cast<E*>(static_cast<char*>(base) + off);
    off += sizeof(E) * (size_t)(count > 0 ? count : 1);
  };
  const int64_t T = a.T;
  take(a.G_ref, 12 * T);
  take(a.G_cur, 12 * T);
  take(a.pts, a.total);
  take(a.sd, 6 * a.S);
  take(a.ref, a.S);
  take(a.pd, a.S);
  take(a.chains, a.ref_order ? T * ICT_EVAL_NQ * 2 * a.eigen_packet : 0);
  take(a.partials, a.ref_order ? 0 : nchunks * ICT_EVAL_NQ);
  take(a.nvis, T);
  take(a.out_H, 36 * T);
  take(a.out_jtr, 6 * T);
  take(a.out_dp, 6 * T);
  take(a.out_ssr, T);
  take(a.pt_ssr, a.total);
  return off;
}

size_t evaluate_poses_workspace(EvalArgs& a, EvalPoses& b, int64_t nchunks, void* base) {
  size_t off = evaluate_workspace(a, nchunks, base);
  a.out_jtr = a.out_dp = a.out_ssr = a.pt_ssr = nullptr;   // the template pass writes H and the factorisation only
  auto take = [&](auto*& p, int64_t count) {
    using E = std::remove_reference_t<decltype(*p)>;
    off = (off + 255) & ~(size_t)255;
    if (base) p = reinterpret_cast<E*>(static_cast<char*>(base) + off);
    off += sizeof(E) * (size_t)(count > 0 ? count : 1);
  };
  const int64_t TK = (int64_t)a.T * b.K;
  take(a.lu, a.T);
  take(b.G_cand, 12 * TK);
  take(b.cand, a.total * b.K);
  take(b.chains, a.ref_order ? TK * EVP_NQ * 2 * a.eigen_packet : 0);
  take(b.partials, a.ref_order ? 0 : nchunks * b.K * EVP_NQ);
  take(b.nvis, TK);
  take(b.out_jtr, 6 * TK);
  take(b.out_dp, 6 * TK);
  take(b.out_ssr, TK);
  return off;
}

// SetPose poses, the points' placements, the template and sd of every pixel slot
static void launch_eval_template(const EvalArgs& a, cudaStream_t st) {
  count_launch();
  k_eval_pose<<<(unsigned)((a.T + 127) / 128), 128, 0, st>>>(a);
  if (a.total > 0) {
    for (int k = 0; k < 2; ++k) count_launch();
    k_eval_points<<<(unsigned)((a.total + 255) / 256), 256, 0, st>>>(a);
    k_eval_slots<<<(unsigned)((a.S + 255) / 256), 256, 0, st>>>(a);
  }
}

// the 28 sums of every track, then its factorisation and solve
static void launch_eval_sums(const EvalArgs& a, int64_t nchunks, cudaStream_t st) {
  const int64_t T = a.T;
  const unsigned solve_blocks = (unsigned)((T + 3) / 4);
  count_launch();                                 // the sums
  if (a.ref_order || nchunks > 0) count_launch();  // the solve
  if (a.ref_order) {
    const int64_t nthr = T * ICT_EVAL_NQ * 2 * a.eigen_packet;
    if (a.eigen_packet == 8) {
      k_eval_chains<8><<<(unsigned)((nthr + 255) / 256), 256, 0, st>>>(a);
      k_eval_solve<8, true><<<solve_blocks, 128, 0, st>>>(a);
    } else {
      k_eval_chains<4><<<(unsigned)((nthr + 255) / 256), 256, 0, st>>>(a);
      k_eval_solve<4, true><<<solve_blocks, 128, 0, st>>>(a);
    }
  } else {
    if (nchunks > 0) k_eval_partials<<<(unsigned)nchunks, 256, 0, st>>>(a);
    k_eval_solve<4, false><<<solve_blocks, 128, 0, st>>>(a);
  }
}

cudaError_t launch_evaluate(const EvalArgs& a, int64_t nchunks, cudaStream_t st) {
  if (a.T <= 0) return cudaSuccess;
  launch_eval_template(a, st);
  if (a.total > 0) {
    count_launch();
    if (a.eigen_packet == 8)
      k_eval_patch<8><<<(unsigned)((a.total + 127) / 128), 128, 0, st>>>(a);
    else
      k_eval_patch<4><<<(unsigned)((a.total + 127) / 128), 128, 0, st>>>(a);
  }
  launch_eval_sums(a, nchunks, st);
  return cudaGetLastError();
}

int64_t evaluate_chunks(int64_t pixels) { return (pixels + ICT_EVAL_CHUNK - 1) / ICT_EVAL_CHUNK; }

template <int W>
static cudaError_t launch_poses_w(const EvalArgs& a, const EvalPoses& b, int64_t nchunks, cudaStream_t st) {
  const int64_t TK = (int64_t)a.T * b.K, ng = (b.K + EVP_KG - 1) / EVP_KG;
  // per track: the template with its mean subtracted, H and its factorisation (a.p_cur is null: G_cur = G_ref, and
  // the J^T r, SSR and visible count of that pass are neither kept nor read)
  launch_eval_template(a, st);
  if (a.total > 0) {
    count_launch();
    k_evp_template<W><<<(unsigned)((a.total + 127) / 128), 128, 0, st>>>(a);
  }
  launch_eval_sums(a, nchunks, st);
  // per candidate
  count_launch();
  k_evp_pose<<<(unsigned)((TK + 127) / 128), 128, 0, st>>>(a, b);
  if (a.total > 0) {
    count_launch();
    const dim3 grid((unsigned)((a.total + 255) / 256), (unsigned)(b.K < 65535 ? b.K : 65535));
    k_evp_points<W><<<grid, 256, 0, st>>>(a, b);
  }
  if (a.ref_order) {
    count_launch();
    k_evp_chains<W><<<(unsigned)((a.T * ng * 2 * W + 255) / 256), 256, 0, st>>>(a, b);
  } else if (nchunks > 0) {
    count_launch();
    k_evp_partials<<<(unsigned)(nchunks * ng), 256, 0, st>>>(a, b);
  }
  count_launch();
  if (a.ref_order)
    k_evp_solve<W, true><<<(unsigned)((TK + 127) / 128), 128, 0, st>>>(a, b);
  else
    k_evp_solve<W, false><<<(unsigned)((TK + 127) / 128), 128, 0, st>>>(a, b);
  return cudaGetLastError();
}

cudaError_t launch_evaluate_poses(const EvalArgs& a, const EvalPoses& b, int64_t nchunks, cudaStream_t st) {
  if (a.T <= 0) return cudaSuccess;
  const int64_t ng = (b.K + EVP_KG - 1) / EVP_KG;
  if (nchunks * ng > 0x7fffffff || a.T * ng * 2 * a.eigen_packet / 256 > 0x7fffffff)
    return cudaErrorInvalidConfiguration;
  return a.eigen_packet == 8 ? launch_poses_w<8>(a, b, nchunks, st) : launch_poses_w<4>(a, b, nchunks, st);
}

}  // namespace ict
