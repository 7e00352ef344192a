// ict_kernels_big.cu — the multi-CTA form of SetPose + TrackPose for ONE track that is too large for a CTA's shared
// memory (dense full-frame alignment: psz = 1, one point per pixel, BASELINE config 4; more than 240 8x8 patches).
//
// Same arithmetic as k_track (ict_kernels.cu), including the optional reference-order sums (sum_mode 1: Hessian and
// J^T r by one CTA running Eigen's eight sequential chains, sixteen with 8-float packets); the template (pat_ref, pat_dx, pat_dy) and the per-point state
// live in a global work buffer that fits the 126 MB L2 for a 1080p frame, reductions are two-stage with a fixed
// order (thread-strided partials -> warp tree -> CTA partial -> one finishing CTA), and the iteration loop is a
// fixed sequence of launches whose kernels return immediately once the on-device convergence flag drops, so
// there is still no host round-trip inside TrackPose.
#include "ict_kernels.cuh"
#include "ict_device.cuh"

#include <type_traits>

namespace ict {

struct BigState {
  float G[12];
  float p[6];
  Lu6 lu;                   // before the first level: lu.lu[0..11] = the template's pose (track_setpose_from)
  float normdp, normdp_init;
  int cont, it, nvis, trace_n, level_it;
  unsigned ticket;          // CTAs that have published their partial sums in the running fused-iteration launch
  long long npix;
};

struct BigWork {
  BigState* st;
  float *ref, *gx, *gy, *pnew;
  float *coef, *w, *mean, *Xc, *Yc, *Zc;
  int *base, *vis;
  float* part;      // [ncta][21]
  float* prod;      // reference-order sums: product arrays, chain-major — prod[(q*NCH + c)*cstride + j] = value of
                    // quantity q at element e = NCH j + c (the elements of Eigen's chain c, contiguous; big_prod_idx), NCH
                    // = 8 chains per sum for 4-float packets, 16 for 8-float packets
  long long cstride;   // floats per chain row of prod (a multiple of the chunk)
  int ncta;
};

#define BIG_CHUNK 2048         /* chain elements per staged chunk (8 KB per chain, 64 KB per stage) of the reference-order
                                  chain kernel: every chunk costs ~150 cycles of hand-over on the critical path, so few and
                                  large ones (512 x 4 stages: 0.66 ms per pass of 247 k additions; 2048 x 2: 0.585 ms) */
#define BIG_STAGES 2
// A stage holds 8 * BIG_CHUNK floats whatever the chain count: sixteen chains (8-float packets) take chunks of half the
// length, and their chains are half as long, so the hand-overs per chain pass stay the same.
__host__ __device__ constexpr int big_chunk(int nch) { return 8 * BIG_CHUNK / nch; }
// row stride of a chain-kernel stage in shared memory: sixteen chains' rows get a 16-byte skew (see k_big_chains)
__host__ __device__ constexpr int big_row_stride(int nch) { return nch == 8 ? big_chunk(nch) : big_chunk(nch) + 4; }
// position of element j of chain c of product row q: chunk-major — the NCH chains' pieces of one chunk are contiguous
// (64 KB), so that a stage of the chain kernel is one stretch of memory
template <int NCH>
__host__ __device__ __forceinline__ long long big_prod_idx(int q, int c, long long j, long long cstride) {
  constexpr int CH = big_chunk(NCH);
  return (long long)q * NCH * cstride + ((j / CH) * NCH + c) * CH + (j % CH);
}
static long long big_cstride(int64_t Nfull, int nch) {
  const long long nj = (Nfull + nch - 1) / nch, ch = big_chunk(nch);
  return ((nj + ch - 1) / ch) * ch;
}

static int big_ncta(int64_t E) {
  // at most four 256-thread CTAs per SM (the streaming kernels use up to 64 registers): one resident wave, no tail.
  // The grid fixes the partition of the two-stage sums, so every kernel of this file uses the same one.
  int64_t c = (E + 1023) / 1024;
  if (c > 148 * 4) c = 148 * 4;
  if (c < 1) c = 1;
  return (int)c;
}

size_t bigtrack_work_bytes(const ict_optparam& op, int64_t npts, int eigen_packet, void* base, BigWork* out) {
  const int64_t P = npts < op.maxpttrack ? npts : op.maxpttrack;
  const int64_t E = P * op.novals;
  const int nch = eigen_packet == 8 ? 16 : 8;
  BigWork w = {};
  w.ncta = big_ncta(E);
  w.cstride = big_cstride((int64_t)op.maxpttrack * op.novals, nch);
  size_t off = 0;
  auto take = [&](auto*& p, int64_t count) {   // 256-byte aligned regions, in this order
    using T = std::remove_reference_t<decltype(*p)>;
    off = (off + 255) & ~(size_t)255;
    if (base) p = reinterpret_cast<T*>(static_cast<char*>(base) + off);
    off += sizeof(T) * (size_t)count;
  };
  take(w.st, 1);
  take(w.ref, E);
  take(w.gx, E);
  take(w.gy, E);
  take(w.pnew, E);
  take(w.coef, 10 * P);
  take(w.w, 4 * P);
  take(w.mean, P);
  take(w.Xc, P);
  take(w.Yc, P);
  take(w.Zc, P);
  take(w.base, P);
  take(w.vis, P);
  take(w.part, 21 * w.ncta);
  take(w.prod, nch * 24 * w.cstride);   // 24 product rows: the 21 Hessian sums at once
  if (out) *out = w;
  return (off + 255) & ~(size_t)255;
}

struct BigArgs {
  TrackParams prm;
  BigWork w;
  int t;
  int n_in, P;
  long long E;
};

// fixed-order CTA reduction of NV per-thread values into part[blockIdx.x*21 + k]
template <int NV>
__device__ __forceinline__ void cta_partials(float* acc, float* part) {
  __shared__ float s_p[8 * 21];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const float v = warp_sum(acc[k]);
    if (lane == 0) s_p[warp * 21 + k] = v;
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    float s = s_p[threadIdx.x];
    for (int wv = 1; wv < nw; ++wv) s = s + s_p[wv * 21 + threadIdx.x];
    part[blockIdx.x * 21 + threadIdx.x] = s;
  }
}

// sum of the CTA partials, fixed order: 256 strided chains -> warp tree -> 8 warps
template <int NV>
__device__ __forceinline__ void finish_partials(const float* part, int ncta, float* out /*shared, NV*/) {
  __shared__ float s_p[8 * 21];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  // a thread's first three CTAs are loaded before the first addition: one L2 round trip for the usual grid
  // (at most 592 CTAs), not one per value
  const int c0 = threadIdx.x, c1 = c0 + blockDim.x, c2 = c1 + blockDim.x;
  float v0[NV], v1[NV], v2[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    v0[k] = c0 < ncta ? __ldcg(part + c0 * 21 + k) : 0.0f;
    v1[k] = c1 < ncta ? __ldcg(part + c1 * 21 + k) : 0.0f;
    v2[k] = c2 < ncta ? __ldcg(part + c2 * 21 + k) : 0.0f;
  }
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    float s = 0.0f;
    if (c0 < ncta) s = s + v0[k];
    if (c1 < ncta) s = s + v1[k];
    if (c2 < ncta) s = s + v2[k];
    for (int c = c2 + blockDim.x; c < ncta; c += blockDim.x) s = s + __ldcg(part + c * 21 + k);
    s = warp_sum(s);
    if (lane == 0) s_p[warp * 21 + k] = s;
  }
  __syncthreads();
  if (threadIdx.x < NV) {
    float s = s_p[threadIdx.x];
    for (int wv = 1; wv < nw; ++wv) s = s + s_p[wv * 21 + threadIdx.x];
    out[threadIdx.x] = s;
  }
  __syncthreads();
}

// ---- per-element work shared by the kernels below --------------------------------------------------------------------
// a pyramid level's intrinsics and image bounds
struct LevelCam {
  float fx, fy, cx, cy, swo, sho;
  int width;
};
__device__ __forceinline__ LevelCam level_cam(const CamLevels& cam, int sl) {
  return {cam.fx[sl], cam.fy[sl], cam.cx[sl], cam.cy[sl], cam.swo[sl], cam.sho[sl], cam.width[sl]};
}

// camera-frame point (x, y, z) projected at level lc: false outside [0, swo] x [0, sho] (odometer.cpp:273-275,
// 369-371), else true with q = the placement of its patch
__device__ __forceinline__ bool project_place(const LevelCam& lc, int pszd2, float x, float y, float z, PatchPlace& q) {
  const float mx = (x / z) * lc.fx + lc.cx;
  const float my = (y / z) * lc.fy + lc.cy;
  if (!((mx >= 0) & (my >= 0) & (mx <= lc.swo) & (my <= lc.sho))) return false;
  q = patch_place(mx, my, pszd2, lc.width);
  return true;
}

__device__ __forceinline__ float sample(const float* __restrict__ img, const PatchPlace& q, int width) {
  return bilin4(img, q.base, width, q.w0, q.w1, q.w2, q.w3);
}

// point i's placement into the per-point arrays (base, w), and back moved to pixel slot e = (i, row r, column c)
__device__ __forceinline__ void store_place(const BigArgs& a, long long i, const PatchPlace& q) {
  a.w.base[i] = q.base;
  a.w.w[i] = q.w0; a.w.w[a.P + i] = q.w1; a.w.w[2LL * a.P + i] = q.w2; a.w.w[3LL * a.P + i] = q.w3;
}
__device__ __forceinline__ PatchPlace slot_place(const BigArgs& a, long long e, long long i, int width) {
  const int n = a.prm.op.novals, psz = a.prm.op.psz;
  const int rem = (int)(e - i * n), r = rem / psz, c = rem - r * psz;
  return {a.w.base[i] + r * width + c, a.w.w[i], a.w.w[a.P + i], a.w.w[2LL * a.P + i], a.w.w[3LL * a.P + i]};
}

// the six steepest-descent values of a slot of point i with gradient (gx, gy), from the point's coefficient rows
// (sd_values' arithmetic)
__device__ __forceinline__ void slot_sd(const BigArgs& a, long long i, float gx, float gy, float* sd) {
  const float* cf = a.w.coef;
  sd[0] = gx * cf[0 * (long long)a.P + i];
  sd[1] = gy * cf[1 * (long long)a.P + i];
  sd[2] = gx * cf[2 * (long long)a.P + i] + gy * cf[3 * (long long)a.P + i];
  sd[3] = gx * cf[4 * (long long)a.P + i] + gy * cf[5 * (long long)a.P + i];
  sd[4] = gx * cf[6 * (long long)a.P + i] + gy * cf[7 * (long long)a.P + i];
  sd[5] = gx * cf[8 * (long long)a.P + i] + gy * cf[9 * (long long)a.P + i];
}

// acc[k] += sd_p * sd_q for the 21 pairs p <= q in ComputeHessian's order
__device__ __forceinline__ void add_hessian(float* acc, const float* sd) {
  int k = 0;
#pragma unroll
  for (int p = 0; p < 6; ++p)
#pragma unroll
    for (int q = p; q < 6; ++q) { acc[k] = acc[k] + sd[p] * sd[q]; ++k; }
}

// ---- the start of a level and the serial tail of a non-fused iteration -----------------------------------------------
// Called by one warp once the level's 21 Hessian sums are in s_H: factors H, resets the level's state and records 0
// iterations for it (a level the stop rule does not enter keeps that count).
__device__ __forceinline__ void big_level_start(const BigArgs& a, int sl, const float* s_H) {
  BigState* S = a.w.st;
  lu6_factor_warp(s_H, S->lu);
  if (threadIdx.x == 0) {
    const ict_optparam& op = a.prm.op;
    S->normdp_init = 1e-10f;
    S->normdp = 1e-10f;
    S->it = 0;
    S->nvis = 0;
    S->cont = keep_iterating(op, 0, 1e-10f, 1e-10f);
    store_level_iters(a.prm.iters, op, a.t, sl, 0);
  }
}

// Solve, pose update, trace record, pixel-residual count, the level's iteration count and the stop rule of one
// iteration of the non-fused paths (one thread); sum6 = the six sums of J^T r.  The same steps as the fused dense
// path's tail in dense_iter_finish, which keeps its own copy: there the state comes from a shared-memory snapshot and
// teacher forcing applies.
__device__ __forceinline__ void big_iter_finish_serial(const BigArgs& a, int sl, const float* sum6) {
  BigState* S = a.w.st;
  const ict_optparam& op = a.prm.op;
  float sumsd[6], dp[6];
  for (int k = 0; k < 6; ++k) sumsd[k] = sum6[k];
  lu6_solve_exact(S->lu, sumsd, dp);   // == lu6_solve, straight-line
  for (int k = 0; k < 6; ++k) S->p[k] += dp[k];
  se3_exp<float>(S->G, S->p);
  const float normdp = normdp_l1(dp);
  if (S->it == 0) S->normdp_init = normdp;
  S->normdp = normdp;
  if (a.prm.trace && S->trace_n < a.prm.trace_cap)
    trace_record(track_trace(a.prm, a.t) + (int64_t)ICT_TRACE_FLOATS * S->trace_n++, sl, S->it, sumsd, dp, normdp, S->nvis);
  S->npix += (long long)S->nvis * op.novals;
  S->nvis = 0;
  S->it += 1;
  store_level_iters(a.prm.iters, op, a.t, sl, S->it);
  S->cont = keep_iterating(op, S->it, S->normdp, S->normdp_init);
}

__global__ void k_big_init(const BigArgs a, int fused) {
  // ResetOdometer for the element/point state + setpose_se3.  The fused dense path keeps (ref, sd1..6) only.
  const long long gid = blockIdx.x * (long long)blockDim.x + threadIdx.x, gsz = (long long)gridDim.x * blockDim.x;
  for (long long e = gid; e < a.E; e += gsz) {
    a.w.ref[e] = 0.0f;
    if (!fused) { a.w.gx[e] = 0.0f; a.w.gy[e] = 0.0f; }
  }
  const int ncoef = fused ? 6 : 10;
  for (long long i = gid; i < a.P; i += gsz) {
    if (!fused) a.w.vis[i] = 0;
    for (int k = 0; k < ncoef; ++k) a.w.coef[(long long)k * a.P + i] = 0.0f;
  }
  if (gid == 0) {
    BigState* S = a.w.st;
    const ict_optparam& op = a.prm.op;
    track_setpose_from(a.prm, a.prm.p_in, a.t, op.donorm != 0, S->p, S->G, S->lu.lu);
    S->npix = 0;
    S->nvis = 0;
    S->trace_n = 0;
    S->cont = 0;
    S->it = 0;
    S->ticket = 0;
  }
}

__global__ void k_big_project_ref(const BigArgs a) {
  const BigState* S = a.w.st;
  const int64_t off = a.prm.pt_off[a.t];
  const float* q = a.prm.pt3d + 3 * off;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.P; i += (long long)gridDim.x * blockDim.x)
    save_rotated_point(a.prm, S->lu.lu, off, a.n_in, i, q[i], q[a.n_in + i], q[2 * (int64_t)a.n_in + i], a.w.Xc, a.w.Yc,
                       a.w.Zc);
}

__global__ void k_big_level_points(const BigArgs a, int sl) {
  const LevelCam lc = level_cam(a.prm.cam, sl);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.P; i += (long long)gridDim.x * blockDim.x) {
    const float xc = a.w.Xc[i], yc = a.w.Yc[i], zc = a.w.Zc[i];
    PatchPlace q;
    if (!project_place(lc, a.prm.op.pszd2, xc, yc, zc, q)) {
      a.w.vis[i] = 0;
    } else {
      a.w.vis[i] = 1;
      store_place(a, i, q);
      float c[10];
      sd_coefs(xc, yc, zc, lc.fx, lc.fy, c);
      for (int k = 0; k < 10; ++k) a.w.coef[(long long)k * a.P + i] = c[k];
    }
  }
}

__global__ void __launch_bounds__(256) k_big_level_gather(const BigArgs a, int sl) {
  const int n = a.prm.op.novals, width = a.prm.cam.width[sl];
  const int rf = a.prm.fixed_ref;
  const float* __restrict__ Iref = a.prm.frames[rf].I[sl];
  const float* __restrict__ Dxr = a.prm.frames[rf].dx[sl];
  const float* __restrict__ Dyr = a.prm.frames[rf].dy[sl];
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < a.E; e += (long long)gridDim.x * blockDim.x) {
    const long long i = e / n;
    if (a.w.vis[i] & 1) {
      const PatchPlace q = slot_place(a, e, i, width);
      a.w.ref[e] = sample(Iref, q, width);
      a.w.gx[e] = sample(Dxr, q, width);
      a.w.gy[e] = sample(Dyr, q, width);
    }
  }
}

// mean subtraction of each visible patch of buf: one warp per patch, fixed order (a warp tree; with exact = 4 or 8 the
// reference's order for that packet width, tmp.sum() of utilities.cpp:112, summed by one lane)
__global__ void k_big_patch_means(const BigArgs a, float* buf, int visbit, int subtract, int exact) {
  const int n = a.prm.op.novals;
  const int lane = threadIdx.x & 31;
  const long long wid = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  for (long long i = wid; i < a.P; i += nwarps) {
    if (!(a.w.vis[i] & visbit)) continue;
    float s = 0.0f;
    if (exact) {
      const float* b = buf + i * n;
      if (lane == 0)
        s = exact == 8 ? eigen_sum_serial<8>([&](int e) { return b[e]; }, n) : eigen_sum_serial<4>([&](int e) { return b[e]; }, n);
    } else {
      for (int k = lane; k < n; k += 32) s = s + buf[i * n + k];
      s = warp_sum(s);
    }
    s = __shfl_sync(0xffffffffu, s, 0);
    const float m = s / n;
    if (lane == 0) a.w.mean[i] = m;
    if (subtract)
      for (int k = lane; k < n; k += 32) buf[i * n + k] = buf[i * n + k] - m;
  }
}

__global__ void __launch_bounds__(256) k_big_level_hessian(const BigArgs a) {
  const int n = a.prm.op.novals;
  float acc[21];
#pragma unroll
  for (int k = 0; k < 21; ++k) acc[k] = 0.0f;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < a.E; e += (long long)gridDim.x * blockDim.x) {
    float sd[6];
    slot_sd(a, e / n, a.w.gx[e], a.w.gy[e], sd);
    add_hessian(acc, sd);
  }
  cta_partials<21>(acc, a.w.part);
}

// (griddepcontrol.*: no-ops unless the launch carries the programmatic-dependent-launch attribute, as the fused dense
// path's launches do — the kernel then becomes resident while its predecessor drains, and lets its successor do so)
__global__ void __launch_bounds__(256) k_big_level_finish(const BigArgs a, int sl) {
  __shared__ float s_H[21];
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  finish_partials<21>(a.w.part, a.w.ncta, s_H);
  if (threadIdx.x < 32) big_level_start(a, sl, s_H);
}

__global__ void k_big_iter_points(const BigArgs a, int sl) {
  BigState* S = a.w.st;
  if (!S->cont) return;
  const LevelCam lc = level_cam(a.prm.cam, sl);
  const int64_t off = a.prm.pt_off[a.t];
  const float* q = a.prm.pt3d + 3 * off;
  int cnt = 0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.P; i += (long long)gridDim.x * blockDim.x) {
    float tx, ty, tz;
    rigid_apply<float>(S->G, q[i], q[a.n_in + i], q[2 * (int64_t)a.n_in + i], tx, ty, tz);
    PatchPlace pp;
    if (!project_place(lc, a.prm.op.pszd2, tx, ty, tz, pp)) {
      a.w.vis[i] &= ~2;
    } else {
      a.w.vis[i] |= 2;
      store_place(a, i, pp);
      ++cnt;
    }
  }
  // integer count: order-independent
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_down_sync(0xffffffffu, cnt, o);
  if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(&S->nvis, cnt);
}

__global__ void __launch_bounds__(256) k_big_iter_sample(const BigArgs a, int sl) {
  if (!a.w.st->cont) return;
  const int n = a.prm.op.novals, width = a.prm.cam.width[sl];
  const float* __restrict__ Inew = a.prm.frames[a.prm.fixed_new].I[sl];
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < a.E; e += (long long)gridDim.x * blockDim.x) {
    const long long i = e / n;
    if (a.w.vis[i] & 2) a.w.pnew[e] = sample(Inew, slot_place(a, e, i, width), width);
  }
}

template <bool PN>
__global__ void __launch_bounds__(256) k_big_iter_elems(const BigArgs a, int sl) {
  if (!a.w.st->cont) return;
  const int n = a.prm.op.novals, width = a.prm.cam.width[sl];
  const float* __restrict__ Inew = a.prm.frames[a.prm.fixed_new].I[sl];
  float acc[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) acc[k] = 0.0f;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < a.E; e += (long long)gridDim.x * blockDim.x) {
    const long long i = e / n;
    if (a.w.vis[i] & 2) {
      float pn;
      if (PN) pn = a.w.pnew[e];   // mean already subtracted by k_big_patch_means
      else pn = sample(Inew, slot_place(a, e, i, width), width);
      const float pd = a.w.ref[e] - pn;
      float cf[10], sd[6];
#pragma unroll
      for (int k = 0; k < 10; ++k) cf[k] = a.w.coef[(long long)k * a.P + i];
      sd_values(a.w.gx[e], a.w.gy[e], cf, sd);
#pragma unroll
      for (int k = 0; k < 6; ++k) acc[k] = acc[k] + sd[k] * pd;
    }
  }
  cta_partials<6>(acc, a.w.part);
}

__global__ void __launch_bounds__(256) k_big_iter_finish(const BigArgs a, int sl, int ncta) {
  BigState* S = a.w.st;
  if (!S->cont) return;
  __shared__ float s_sum[21];
  if (ncta == 1) {   // reference-order sums were completed by k_big_chains: take them as they are
    if (threadIdx.x < 6) s_sum[threadIdx.x] = a.w.part[threadIdx.x];
    __syncthreads();
  } else {
    finish_partials<6>(a.w.part, ncta, s_sum);
  }
  if (threadIdx.x == 0) big_iter_finish_serial(a, sl, s_sum);
}

// ---- reference-order (sum_mode 1) variants -----------------------------------------------------------------------------
// ---- reference-order sums over arrays too long for one thread per chain -----------------------------------------------
// Eigen's chain c of a sum adds the elements c, c+8, c+16, ... one after the other: 4 cycles per addition whatever
// else happens, so a sum over E elements costs E/2 cycles at best (1 M cycles = 0.5 ms for a 1080p dense template).
// The first form of this path ran each chain as one thread fetching its operands from five global arrays as it went
// (~2500 cycles per element: 12.5 s per dense TrackPose).  Now in two phases:
//   1. k_big_products (all SMs, streaming): the values to be summed — sd_k * pdiff for the six J^T r sums, sd_a * sd_b
//      for six of the 21 Hessian sums per pass — with the reference's roundings, written CHAIN-MAJOR (the elements of
//      chain c of quantity q contiguous), so that
//   2. k_big_chains (one warp per quantity, lane c = chain c) streams its NCH rows through a two-stage
//      shared-memory ring with bulk asynchronous copies (cp.async.bulk + mbarrier transaction counts, 64 KB per
//      stage) and does nothing but LDS.128 + four dependent additions per four elements.
// NCH = 8 chains for Eigen's 4-float packets, 16 for 8-float packets.
// Same additions in the same order as eigen_chain: the sums are bit-identical to the one-thread form (tested against
// the oracle on dense alignment and on tracks of 700-900 8x8 patches).
template <int MODE, int NCH>   // MODE 0: iteration (sd_q * pnew); 1: Hessian, pairs 6*pass .. 6*pass+5 of ComputeHessian's order
__global__ void __launch_bounds__(256) k_big_products(const BigArgs a, int pass) {
  if (MODE == 0 && !a.w.st->cont) return;
  const int n = a.prm.op.novals;
  const long long lim = a.E;                       // elements beyond E are zeros the reference adds nothing for
  const long long nj = (lim + NCH - 1) / NCH;
  for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j < nj; j += (long long)gridDim.x * blockDim.x) {
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const long long e = NCH * j + c;
      float v[6];
      if (e < lim) {
        float sd[6];
        slot_sd(a, n == 1 ? e : e / n, a.w.gx[e], a.w.gy[e], sd);
        if (MODE == 0) {
          const float pd = a.w.pnew[e];
#pragma unroll
          for (int q = 0; q < 6; ++q) v[q] = sd[q] * pd;
        } else {
#pragma unroll
          for (int q = 0; q < 6; ++q) {
            const int idx = 6 * pass + q;      // pair (x, y), x <= y, in row-major upper-triangle order
            int x = 0, y = 0, k = 0;
#pragma unroll
            for (int aa = 0; aa < 6; ++aa)
#pragma unroll
              for (int bb = aa; bb < 6; ++bb) { if (k == idx) { x = aa; y = bb; } ++k; }
            float sx = sd[0], sy = sd[0];
#pragma unroll
            for (int m = 1; m < 6; ++m) { sx = x == m ? sd[m] : sx; sy = y == m ? sd[m] : sy; }
            v[q] = idx < 21 ? sx * sy : 0.0f;
          }
        }
#pragma unroll
        for (int q = 0; q < 6; ++q) a.w.prod[big_prod_idx<NCH>((MODE == 1 ? 6 * pass : 0) + q, c, j, a.w.cstride)] = v[q];
      }
    }
  }
}

// Reference order, no patch normalisation: k_big_iter_points + k_big_iter_pdiff + k_big_products<0> in one launch.  Every
// element re-derives its point's projection and placement (the same operations on the same operands: the same bits)
// instead of reading them from per-point arrays written by an earlier launch; the point's first element counts it.
template <int NCH>
__global__ void __launch_bounds__(256) k_big_iter_fused_exact(const BigArgs a, int sl) {
  BigState* S = a.w.st;
  if (!S->cont) return;
  const LevelCam lc = level_cam(a.prm.cam, sl);
  const int width = lc.width, n = a.prm.op.novals, psz = a.prm.op.psz, pszd2 = a.prm.op.pszd2;
  const float* __restrict__ Inew = a.prm.frames[a.prm.fixed_new].I[sl];
  const float* q3 = a.prm.pt3d + 3 * a.prm.pt_off[a.t];
  const long long lim = a.E;
  const long long nj = (lim + NCH - 1) / NCH;
  const float* cf = a.w.coef;
  float G[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) G[k] = S->G[k];
  int cnt = 0;
  for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j < nj; j += (long long)gridDim.x * blockDim.x) {
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const long long e = NCH * j + c;
      if (e < lim) {
        const long long i = n == 1 ? e : e / n;
        const int rem = (int)(e - i * n), r = rem / psz, cc = rem - r * psz;
        const float X = q3[i], Y = q3[a.n_in + i], Z = q3[2 * (int64_t)a.n_in + i];
        float tx, ty, tz;
        rigid_apply(G, X, Y, Z, tx, ty, tz);
        PatchPlace pp;
        float pd = 0.0f;
        if (project_place(lc, pszd2, tx, ty, tz, pp)) {
          pd = a.w.ref[e] - bilin4(Inew, pp.base + r * width + cc, width, pp.w0, pp.w1, pp.w2, pp.w3);
          if (rem == 0) ++cnt;
        }
        const float gx = a.w.gx[e], gy = a.w.gy[e];
        float sd[6];
        sd[0] = gx * cf[0 * (long long)a.P + i];
        sd[1] = gy * cf[1 * (long long)a.P + i];
        sd[2] = gx * cf[2 * (long long)a.P + i] + gy * cf[3 * (long long)a.P + i];
        sd[3] = gx * cf[4 * (long long)a.P + i] + gy * cf[5 * (long long)a.P + i];
        sd[4] = gx * cf[6 * (long long)a.P + i] + gy * cf[7 * (long long)a.P + i];
        sd[5] = gx * cf[8 * (long long)a.P + i] + gy * cf[9 * (long long)a.P + i];
#pragma unroll
        for (int q = 0; q < 6; ++q) a.w.prod[big_prod_idx<NCH>(q, c, j, a.w.cstride)] = sd[q] * pd;
      }
    }
  }
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_down_sync(0xffffffffu, cnt, o);   // integer count: order-independent
  if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(&S->nvis, cnt);
}

// One CTA (one warp) per quantity q < nq.  out[q] = the Eigen-order sum of the quantity's E values (zeros up to
// Nfull), finished like redux_impl::run with the few tail elements re-read from the product rows.
// NCH = 8: lanes 0..7 read rows 8 KB apart — the same banks, but at eight lanes per LDS.128 phase that costs 64 cycles
// per 32 dependent additions (128).  NCH = 16 doubles the lanes and halves the additions, so its rows are staged with
// a 16-byte skew (one bulk copy per row) and the sixteen lanes' reads are conflict-free.
template <int NCH>
__global__ void __launch_bounds__(64) k_big_chains(const BigArgs a, int nq, float* out, int iteration) {
  if (iteration && !a.w.st->cont) return;
  constexpr int CH = big_chunk(NCH);                     // chain elements per stage
  constexpr int RS = big_row_stride(NCH);                // row stride of a stage in shared memory
  extern __shared__ __align__(128) float s_ring[];     // [BIG_STAGES][NCH][RS]
  __shared__ unsigned long long s_full[BIG_STAGES], s_free[BIG_STAGES];
  __shared__ float s_ch[NCH];
  const int q = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (q >= nq) return;
  const int Nfull = a.prm.op.maxpttrack * a.prm.op.novals, E = (int)a.E;
  const int as2 = (Nfull / NCH) * NCH, lim = as2 < E ? as2 : E;
  const float* rows = a.w.prod + (long long)q * NCH * a.w.cstride;
  // chain c has cnt_c = #{e < lim : e % NCH == c} elements; all chains need ceil(lim / NCH) positions at most
  const int njmax = (lim + NCH - 1) / NCH;
  const int nchunk = (njmax + CH - 1) / CH;
  if (threadIdx.x < BIG_STAGES) {
    mbar_init(&s_full[threadIdx.x], 1);
    mbar_init(&s_free[threadIdx.x], 1);
  }
  mbar_fence_init();
  __syncthreads();
  if (warp == 1) {
    // the copy warp: a chunk's NCH rows (contiguous, 64 KB) into stage chunk % BIG_STAGES as soon as the chain warp
    // has released the stage — kept off the chain warp, whose every cycle is on the critical path
    if (lane == 0)
      for (int chunk = 0; chunk < nchunk; ++chunk) {
        const int st = chunk % BIG_STAGES, use = chunk / BIG_STAGES;
        if (use > 0) mbar_wait(&s_free[st], (use - 1) & 1);
        mbar_expect_tx(&s_full[st], (unsigned)(NCH * CH * sizeof(float)));
        const float* src = rows + (long long)chunk * NCH * CH;
        if (RS == CH) {
          bulk_g2s(s_ring + st * NCH * RS, src, (unsigned)(NCH * CH * sizeof(float)), &s_full[st]);
        } else {
          for (int r = 0; r < NCH; ++r)
            bulk_g2s(s_ring + (st * NCH + r) * RS, src + r * CH, (unsigned)(CH * sizeof(float)), &s_full[st]);
        }
      }
    return;
  }
  const int c = lane & (NCH - 1);
  const int cnt = c < lim ? (lim - c + NCH - 1) / NCH : 0;   // this chain's elements
  float acc = -0.0f;                                     // -0 + x == x: the chain starts with its first element
  for (int chunk = 0; chunk < nchunk; ++chunk) {
    const int st = chunk % BIG_STAGES;
    mbar_wait(&s_full[st], (chunk / BIG_STAGES) & 1);
    if (lane < NCH) {
      const float4* p4 = reinterpret_cast<const float4*>(s_ring + (st * NCH + c) * RS);
      const int have = min(CH, cnt - chunk * CH);       // may be <= 0 for the last chunk of a short chain
      int i = 0;
      if (have >= 32) {
        // 32 elements per trip, the next trip's eight quads loaded ahead of this trip's 32 dependent additions
        float4 v[8], n[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) v[r] = p4[r];
        for (; i + 64 <= have; i += 32) {
#pragma unroll
          for (int r = 0; r < 8; ++r) n[r] = p4[i / 4 + 8 + r];
#pragma unroll
          for (int r = 0; r < 8; ++r) { acc = acc + v[r].x; acc = acc + v[r].y; acc = acc + v[r].z; acc = acc + v[r].w; }
#pragma unroll
          for (int r = 0; r < 8; ++r) v[r] = n[r];
        }
#pragma unroll
        for (int r = 0; r < 8; ++r) { acc = acc + v[r].x; acc = acc + v[r].y; acc = acc + v[r].z; acc = acc + v[r].w; }
        i += 32;
      }
      const float* p1 = reinterpret_cast<const float*>(p4);
      for (; i < have; ++i) acc = acc + p1[i];
    }
    __syncwarp();                                        // every chain lane has read the stage: hand it back
    if (lane == 0) mbar_arrive(&s_free[st]);
  }
  if (lane < NCH) s_ch[lane] = cnt > 0 ? acc : 0.0f;
  __syncwarp();
  if (lane == 0) {
    auto val = [&](int e) { return a.w.prod[big_prod_idx<NCH>(q, e % NCH, e / NCH, a.w.cstride)]; };
    out[q] = eigen_finish<NCH / 2>(s_ch, val, Nfull, E);
  }
}

// the level start after the 21 reference-order Hessian sums (part[0..20]) are in
__global__ void __launch_bounds__(32) k_big_hessian_exact_finish(const BigArgs a, int sl) {
  __shared__ float s_H[21];
  if (threadIdx.x < 21) s_H[threadIdx.x] = a.w.part[threadIdx.x];
  __syncwarp();
  big_level_start(a, sl, s_H);
}

// pdiff of every slot into w.pnew (0 where the point is not visible in the new frame)
template <bool PN>
__global__ void __launch_bounds__(256) k_big_iter_pdiff(const BigArgs a, int sl) {
  if (!a.w.st->cont) return;
  const int n = a.prm.op.novals, width = a.prm.cam.width[sl];
  const float* __restrict__ Inew = a.prm.frames[a.prm.fixed_new].I[sl];
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < a.E; e += (long long)gridDim.x * blockDim.x) {
    const long long i = e / n;
    float pd = 0.0f;
    if (a.w.vis[i] & 2) pd = a.w.ref[e] - (PN ? a.w.pnew[e] : sample(Inew, slot_place(a, e, i, width), width));
    a.w.pnew[e] = pd;
  }
}

// ==================================================================================================
// Fused dense path: psz = 1 (one pixel per point), tree sums, no patch normalisation — BASELINE config 4.
// The general kernels above keep 19 words of per-point state alive between launches (gx, gy, ten coefficients, four
// weights, base, visibility) and need three launches per iteration.  With one pixel per point the six
// steepest-descent values ARE per-point state, so the template is (ref, sd1..sd6) = 28 B per point, an iteration
// streams 40 B per point (X, Y, Z, ref, sd) plus the four gathered texels — the 44 B per pixel-residual of SURVEY.md
// §8(d) — and everything an iteration does fits one launch: project, place, sample, residual, six partial sums per
// CTA, and the CTA that publishes its partials LAST (ticket counter) adds them in the fixed order, solves, updates
// the pose and evaluates the stop rule.  Same per-element arithmetic, same thread partition and same summation order
// as k_big_iter_points/elems/finish: results are bit-identical to that path (tests/test_gpu_parity.py).
// ==================================================================================================
__global__ void __launch_bounds__(256, 4) k_dense_level(const BigArgs a, int sl) {   // 592 CTAs = one resident wave
  const LevelCam lc = level_cam(a.prm.cam, sl);
  const int rf = a.prm.fixed_ref;
  const float* __restrict__ Iref = a.prm.frames[rf].I[sl];
  const float* __restrict__ Dxr = a.prm.frames[rf].dx[sl];
  const float* __restrict__ Dyr = a.prm.frames[rf].dy[sl];
  const long long P = a.P;
  float* sdp = a.w.coef;                   // sd_k of point i at sdp[k * P + i] (the coefficient region, 10 P floats)
  asm volatile("griddepcontrol.wait;" ::: "memory");                // the previous level's iterations are complete
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  float acc[21];
#pragma unroll
  for (int k = 0; k < 21; ++k) acc[k] = 0.0f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < P; i += (long long)gridDim.x * blockDim.x) {
    const float xc = a.w.Xc[i], yc = a.w.Yc[i], zc = a.w.Zc[i];
    float sd[6];
    PatchPlace q;
    if (project_place(lc, a.prm.op.pszd2, xc, yc, zc, q)) {               // util_getPatch_grad, one pixel
      a.w.ref[i] = sample(Iref, q, lc.width);
      const float gx = sample(Dxr, q, lc.width);
      const float gy = sample(Dyr, q, lc.width);
      float c[10];
      sd_coefs(xc, yc, zc, lc.fx, lc.fy, c);
      sd_values(gx, gy, c, sd);                                              // odometer.cpp:317-326
#pragma unroll
      for (int k = 0; k < 6; ++k) sdp[k * P + i] = sd[k];
    } else {                               // out of the reference image: the previous level's values stay (SURVEY §9.6)
#pragma unroll
      for (int k = 0; k < 6; ++k) sd[k] = sdp[k * P + i];
    }
    add_hessian(acc, sd);
  }
  cta_partials<21>(acc, a.w.part);
}

// the new image at the projection of reference point (X, Y, Z) under pose G, one pixel; vis: inside the level
__device__ __forceinline__ float dense_sample(const LevelCam& lc, int pszd2, const float* G, const float* __restrict__ Inew,
                                              float X, float Y, float Z, bool& vis) {
  float tx, ty, tz;
  rigid_apply(G, X, Y, Z, tx, ty, tz);                                         // project_pt, pose.cpp:307-397
  PatchPlace pp;
  vis = project_place(lc, pszd2, tx, ty, tz, pp);
  return vis ? sample(Inew, pp, lc.width) : 0.0f;
}

// Shared tail of the dense iteration kernels: CTA partial sums, visible-point count, ticket; the CTA that arrives last
// adds the partials in the fixed order, solves, updates the pose and evaluates the stop rule.
// L: the state as it was when the launch began (the kernel's shared-memory copy, or S itself): the last CTA's serial
// tail then reads no global memory but the partials.
__device__ __forceinline__ void dense_iter_finish(const BigArgs& a, int sl, float* acc, int cnt, const BigState* L) {
  BigState* S = a.w.st;
  __shared__ float s_sum[8];
  __shared__ int s_cnt[8];
  __shared__ bool s_last;
  // visible points of this CTA (integers: order-independent); published as slot 6 of the CTA's partials
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_down_sync(0xffffffffu, cnt, o);
  if ((threadIdx.x & 31) == 0) s_cnt[threadIdx.x >> 5] = cnt;
  cta_partials<6>(acc, a.w.part);          // (has a CTA barrier before its stores)
  if (threadIdx.x == 6) {
    int c = 0;
    for (int wv = 0; wv < (int)(blockDim.x >> 5); ++wv) c += s_cnt[wv];
    a.w.part[blockIdx.x * 21 + 6] = __int_as_float(c);
  }
  __threadfence();                         // this CTA's partial sums are visible before its ticket is
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(&S->ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!s_last) return;
  // ---- the last CTA: 9a fixed-order sum of the CTA partials, 9b solve, 10 update, stop rule -----------------------
  __threadfence();
  {
    __shared__ float s_p[8 * 8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5, ncta = gridDim.x;
    // same order as finish_partials<6> (per thread: CTAs tid, tid + 256, ... ascending; warp tree; warps ascending);
    // all of a thread's partials are loaded (past L1) before the first addition: one L2 round trip, not eighteen
    float v[3][7];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const int c = threadIdx.x + j * 256;
#pragma unroll
      for (int k = 0; k < 7; ++k) v[j][k] = c < ncta ? __ldcg(a.w.part + c * 21 + k) : 0.0f;
    }
    {
      int nv = 0;
#pragma unroll
      for (int j = 0; j < 3; ++j) nv += __float_as_int(v[j][6]);
      for (int c = threadIdx.x + 768; c < ncta; c += blockDim.x) nv += __float_as_int(__ldcg(a.w.part + c * 21 + 6));
      for (int o = 16; o > 0; o >>= 1) nv += __shfl_down_sync(0xffffffffu, nv, o);
      if (lane == 0) s_cnt[warp] = nv;
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) {
      float sm = 0.0f;
#pragma unroll
      for (int j = 0; j < 3; ++j)
        if (threadIdx.x + j * 256 < ncta) sm = sm + v[j][k];
      for (int c = threadIdx.x + 768; c < ncta; c += blockDim.x) sm = sm + __ldcg(a.w.part + c * 21 + k);
      sm = warp_sum(sm);
      if (lane == 0) s_p[warp * 8 + k] = sm;
    }
    __syncthreads();
    if (threadIdx.x < 6) {
      float sm = s_p[threadIdx.x];
      for (int wv = 1; wv < nw; ++wv) sm = sm + s_p[wv * 8 + threadIdx.x];
      s_sum[threadIdx.x] = sm;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const ict_optparam& op = a.prm.op;
    float sumsd[6], dp[6];
    for (int k = 0; k < 6; ++k) sumsd[k] = s_sum[k];
    lu6_solve_exact(L->lu, sumsd, dp);   // == lu6_solve, straight-line
    float pnew[6];
    const float* tf = nullptr;       // teacher forcing (tests): continue from the oracle's pose
    if (a.prm.teacher && a.prm.trace && L->trace_n < a.prm.trace_cap)
      tf = a.prm.teacher + ((int64_t)a.t * a.prm.trace_cap + L->trace_n) * 8;
    for (int k = 0; k < 6; ++k) { pnew[k] = tf ? tf[k] : L->p[k] + dp[k]; S->p[k] = pnew[k]; }
    se3_exp<float>(S->G, pnew);
    const float normdp = normdp_l1(dp);
    const int it = L->it;
    const float normdp_init = it == 0 ? normdp : L->normdp_init;
    if (it == 0) S->normdp_init = normdp;
    S->normdp = normdp;
    int nvis = 0;
    for (int wv = 0; wv < (int)(blockDim.x >> 5); ++wv) nvis += s_cnt[wv];
    if (a.prm.trace && L->trace_n < a.prm.trace_cap) {
      trace_record(track_trace(a.prm, a.t) + (int64_t)ICT_TRACE_FLOATS * L->trace_n, sl, it, sumsd, dp, normdp, nvis);
      S->trace_n = L->trace_n + 1;
    }
    S->npix = L->npix + (long long)nvis * op.novals;
    S->it = it + 1;
    store_level_iters(a.prm.iters, op, a.t, sl, it + 1);
    S->cont = tf ? (tf[6] != 0.0f) : keep_iterating(op, it + 1, normdp, normdp_init);
    S->ticket = 0;
  }
}

__global__ void __launch_bounds__(256, 4) k_dense_iter(const BigArgs a, int sl) {
  BigState* S = a.w.st;
  if (!S->cont) return;
  __shared__ float s_G[12];
  if (threadIdx.x < 12) s_G[threadIdx.x] = S->G[threadIdx.x];
  __syncthreads();
  float G[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) G[k] = s_G[k];
  const LevelCam lc = level_cam(a.prm.cam, sl);
  const float* __restrict__ Inew = a.prm.frames[a.prm.fixed_new].I[sl];
  const int64_t off = a.prm.pt_off[a.t];
  const float* __restrict__ q = a.prm.pt3d + 3 * off;
  const long long P = a.P;
  const float* __restrict__ sdp = a.w.coef;
  float acc[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) acc[k] = 0.0f;
  int cnt = 0;
  // Two points per trip: both points' streams (X, Y, Z, ref, sd1..6) and then both gathers are in flight together;
  // the additions stay in point order, so the sums are those of the one-point loop.
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < P; i += 2 * stride) {
    const long long j = i + stride;
    const bool hj = j < P;
    const float X0 = q[i], Y0 = q[a.n_in + i], Z0 = q[2 * (int64_t)a.n_in + i];
    const float X1 = hj ? q[j] : 0.0f, Y1 = hj ? q[a.n_in + j] : 0.0f, Z1 = hj ? q[2 * (int64_t)a.n_in + j] : 1.0f;
    const float r0 = a.w.ref[i], r1 = hj ? a.w.ref[j] : 0.0f;
    float s0[6], s1[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) { s0[k] = sdp[k * P + i]; s1[k] = hj ? sdp[k * P + j] : 0.0f; }
    bool v0, v1 = false;
    const float pn0 = dense_sample(lc, a.prm.op.pszd2, G, Inew, X0, Y0, Z0, v0);
    const float pn1 = hj ? dense_sample(lc, a.prm.op.pszd2, G, Inew, X1, Y1, Z1, v1) : 0.0f;
    if (v0) {
      const float pd = r0 - pn0;                                               // pdiff, odometer.cpp:381
#pragma unroll
      for (int k = 0; k < 6; ++k) acc[k] = acc[k] + s0[k] * pd;                 // sd_k_proj and its sum, :386-404
      ++cnt;
    }
    if (hj && v1) {
      const float pd = r1 - pn1;
#pragma unroll
      for (int k = 0; k < 6; ++k) acc[k] = acc[k] + s1[k] * pd;
      ++cnt;
    }
  }
  dense_iter_finish(a, sl, acc, cnt, S);
}

// The same iteration with the five streams of a point (X, Y, Z, ref, sd1..6: 40 B) staged through shared memory by
// bulk asynchronous copies (cp.async.bulk, the copy engine behind TMA) three tiles of 256 points ahead: the DRAM round
// trip of the streams is off the threads' critical path, which keeps only the projection, the placement and the
// four-texel gather (two tiles per trip, for more gathers in flight, was not faster: 35 vs 33 us).  CTA b takes the tiles b, b + G, b + 2G, ... and thread t the point t of each — the partition
// and order of the grid-stride loop above, hence the same sums bit for bit.  Needs 16-byte aligned streams
// (point count a multiple of 4); the launcher falls back to k_dense_iter otherwise.
template <int NST>
__global__ void __launch_bounds__(256, 4) k_dense_iter_tma(const BigArgs a, int sl) {
  BigState* S = a.w.st;
  extern __shared__ __align__(128) unsigned char dense_smem[];
  float (*s_buf)[10][256] = reinterpret_cast<float (*)[10][256]>(dense_smem);
  __shared__ unsigned long long s_full[NST];
  __shared__ BigState s_S;                 // the state when this launch began: pose, LU factors, counters
  const int tid = threadIdx.x;
  // ---- before the previous launch has finished (programmatic dependent launch): nothing here reads what an
  // iteration writes; the streams of the first NST tiles are requested already -------------------------------------
  const int64_t off = a.prm.pt_off[a.t];
  const float* q = a.prm.pt3d + 3 * off;
  const long long P = a.P;
  const float* sdp = a.w.coef;
  const int ntile = (int)((P + 255) / 256);
  const int nmine = ntile > (int)blockIdx.x ? (ntile - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  auto issue = [&](int n) {               // thread 0: the n-th tile of this CTA into stage n % NST
    const long long i0 = ((long long)blockIdx.x + (long long)n * gridDim.x) * 256;
    const unsigned bytes = (unsigned)((P - i0 < 256 ? P - i0 : 256) * 4);
    const int st = n % NST;
    mbar_expect_tx(&s_full[st], 10 * bytes);
    bulk_g2s(s_buf[st][0], q + i0, bytes, &s_full[st]);
    bulk_g2s(s_buf[st][1], q + a.n_in + i0, bytes, &s_full[st]);
    bulk_g2s(s_buf[st][2], q + 2 * (int64_t)a.n_in + i0, bytes, &s_full[st]);
    bulk_g2s(s_buf[st][3], a.w.ref + i0, bytes, &s_full[st]);
#pragma unroll
    for (int k = 0; k < 6; ++k) bulk_g2s(s_buf[st][4 + k], sdp + k * P + i0, bytes, &s_full[st]);
  };
  if (tid == 0) {
    for (int k = 0; k < NST; ++k) mbar_init(&s_full[k], 1);
    mbar_fence_init();
    for (int n = 0; n < NST && n < nmine; ++n) issue(n);
  }
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // the next iteration may become resident as CTAs retire
  asm volatile("griddepcontrol.wait;" ::: "memory");                // the previous launch is complete and visible
  if (tid < (int)(sizeof(BigState) / 4)) reinterpret_cast<int*>(&s_S)[tid] = reinterpret_cast<const int*>(S)[tid];
  __syncthreads();
  if (!s_S.cont) {                         // converged: the requested tiles must land before the CTA may retire
    if (tid == 0)
      for (int n = 0; n < NST && n < nmine; ++n) mbar_wait(&s_full[n], 0);
    return;
  }
  float G[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) G[k] = s_S.G[k];
  const LevelCam lc = level_cam(a.prm.cam, sl);
  const float* __restrict__ Inew = a.prm.frames[a.prm.fixed_new].I[sl];
  float acc[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) acc[k] = 0.0f;
  int cnt = 0;
  // (Tried: placing tile n+1 and issuing its gather before folding tile n — 23.1 instead of 21.3 us per iteration.)
  for (int n = 0; n < nmine; ++n) {
    const int st = n % NST;
    const long long i = ((long long)blockIdx.x + (long long)n * gridDim.x) * 256 + tid;
    mbar_wait(&s_full[st], (n / NST) & 1);
    bool vis = false;
    float pn = 0.0f;
    if (i < P) pn = dense_sample(lc, a.prm.op.pszd2, G, Inew, s_buf[st][0][tid], s_buf[st][1][tid], s_buf[st][2][tid], vis);
    if (vis) {
      const float pd = s_buf[st][3][tid] - pn;                                 // pdiff, odometer.cpp:381
#pragma unroll
      for (int k = 0; k < 6; ++k) acc[k] = acc[k] + s_buf[st][4 + k][tid] * pd;   // sd_k_proj and its sum, :386-404
      ++cnt;
    }
    __syncthreads();                       // every thread has read the stage
    if (tid == 0 && n + NST < nmine) issue(n + NST);
  }
  dense_iter_finish(a, sl, acc, cnt, &s_S);
}

__global__ void k_big_final(const BigArgs a) {
  const BigState* S = a.w.st;
  finish_track(a.prm, a.t, a.prm.op.donorm != 0, S->p, S->G, a.prm.p_out, a.prm.npixres, S->npix,
               track_trace(a.prm, a.t), S->trace_n);
}

// One counted launch of a kernel of this file.  pdl: programmatic stream serialization — the kernel may become resident
// while its predecessor drains, so it has to start with griddepcontrol.wait.
template <typename... KArgs, typename... Args>
static void big_launch(void (*k)(KArgs...), int grid, int threads, size_t smem, bool pdl, cudaStream_t st,
                       Args&&... args) {
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr.val.programmaticStreamSerializationAllowed = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cfg.attrs = &attr;
  cfg.numAttrs = pdl ? 1 : 0;
  cudaLaunchKernelEx(&cfg, k, std::forward<Args>(args)...);
  count_launch();
}

// NCH: chains per reference-order sum (8 for 4-float packets, 16 for 8-float packets)
template <int NCH>
static cudaError_t track_big(const BigArgs& a, cudaStream_t st) {
  const TrackParams& prm = a.prm;
  const ict_optparam& op = prm.op;
  const int ncta = a.w.ncta;
  const int pcta_ = (int)((a.P + 255) / 256 < 148 * 8 ? (a.P + 255) / 256 : 148 * 8);
  const int pcta = pcta_ > 0 ? pcta_ : 1;   // an empty track still runs the launch chain (its sums are empty, its pose unchanged)
  const bool pn = op.dopatchnorm != 0;
  const bool ex = prm.sum_mode != 0;   // reference-order sums
  const bool fused = !pn && !ex && !prm.force_general && op.novals == 1;
  const int mean_order = ex ? prm.eigen_packet : 0;
  constexpr size_t chain_smem = sizeof(float) * BIG_STAGES * NCH * big_row_stride(NCH);   // 128 KB; 128.5 KB for NCH 16
  if (ex) {
    const cudaError_t e = set_kernel_attrs<k_big_chains<NCH>>((int)chain_smem, -1);
    if (e != cudaSuccess) return e;
  }
  // bulk-copy staging needs 16-byte aligned streams: point counts and the track's offset multiples of four
  const bool tma = a.t == 0 && (a.P % 4 == 0) && (a.n_in % 4 == 0);   // t == 0: offset 0
  big_launch(k_big_init, ncta, 256, 0, false, st, a, fused ? 1 : 0);
  big_launch(k_big_project_ref, pcta, 256, 0, false, st, a);
  for (int sl = op.lv_f; sl >= op.lv_l; --sl) {
    // the level's template and Hessian, then its start (factorisation, state)
    if (fused) {   // programmatic dependent launches: each kernel becomes resident while its predecessor drains
      big_launch(k_dense_level, ncta, 256, 0, true, st, a, sl);
      big_launch(k_big_level_finish, 1, 256, 0, true, st, a, sl);
    } else {
      big_launch(k_big_level_points, pcta, 256, 0, false, st, a, sl);
      big_launch(k_big_level_gather, ncta, 256, 0, false, st, a, sl);
      if (pn) big_launch(k_big_patch_means, pcta, 256, 0, false, st, a, a.w.ref, 1, 1, mean_order);
      if (ex) {
        // the products of all 21 sums (four passes of six rows), then their 21 x NCH chains side by side: one chain
        // pass (E / NCH dependent additions) per level instead of four
        for (int pass = 0; pass < 4; ++pass) big_launch(k_big_products<1, NCH>, ncta, 256, 0, false, st, a, pass);
        big_launch(k_big_chains<NCH>, 21, 64, chain_smem, false, st, a, 21, a.w.part, 0);
        big_launch(k_big_hessian_exact_finish, 1, 32, 0, false, st, a, sl);
      } else {
        big_launch(k_big_level_hessian, ncta, 256, 0, false, st, a);
        big_launch(k_big_level_finish, 1, 256, 0, false, st, a, sl);
      }
    }
    for (int it = 0; it < op.maxiter; ++it) {
      if (fused) {
        // one launch per iteration; with programmatic dependent launch, iteration k+1 becomes resident while the last
        // CTA of iteration k still runs the solve, and its first tiles are in flight by the time the pose is published.
        // k_dense_iter has no griddepcontrol.wait, so it is launched in stream order.
        if (tma) big_launch(k_dense_iter_tma<3>, ncta, 256, 3 * 10240, true, st, a, sl);
        else big_launch(k_dense_iter, ncta, 256, 0, false, st, a, sl);
      } else if (ex && !pn && a.E <= (1 << 18)) {
        // three launches per iteration instead of five: products of all elements, the chains, the serial tail.  For
        // tracks whose launches are latency-bound; beyond ~256 k elements the three streaming kernels below are faster
        // than the fused one.  (The serial tail inside the chain kernel's last CTA was measured: passing the argument
        // block on costs the chain kernel a local copy of it, 26 -> 32 ms per dense TrackPose.)
        big_launch(k_big_iter_fused_exact<NCH>, ncta, 256, 0, false, st, a, sl);
        big_launch(k_big_chains<NCH>, 6, 64, chain_smem, false, st, a, 6, a.w.part, 1);
        big_launch(k_big_iter_finish, 1, 256, 0, false, st, a, sl, 1);
      } else {
        big_launch(k_big_iter_points, pcta, 256, 0, false, st, a, sl);
        if (pn) {
          big_launch(k_big_iter_sample, ncta, 256, 0, false, st, a, sl);
          big_launch(k_big_patch_means, pcta, 256, 0, false, st, a, a.w.pnew, 2, 1, mean_order);
        }
        if (ex) {
          big_launch(pn ? k_big_iter_pdiff<true> : k_big_iter_pdiff<false>, ncta, 256, 0, false, st, a, sl);
          big_launch(k_big_products<0, NCH>, ncta, 256, 0, false, st, a, 0);
          big_launch(k_big_chains<NCH>, 6, 64, chain_smem, false, st, a, 6, a.w.part, 1);
        } else {
          big_launch(pn ? k_big_iter_elems<true> : k_big_iter_elems<false>, ncta, 256, 0, false, st, a, sl);
        }
        big_launch(k_big_iter_finish, 1, 256, 0, false, st, a, sl, ex ? 1 : ncta);
      }
    }
  }
  big_launch(k_big_final, 1, 1, 0, false, st, a);
  return cudaGetLastError();
}

cudaError_t launch_track_big(const TrackParams& prm, int t, int64_t npts, void* work, cudaStream_t st) {
  BigArgs a;
  a.prm = prm;
  bigtrack_work_bytes(prm.op, npts, prm.eigen_packet, work, &a.w);
  a.t = t;
  a.n_in = (int)npts;
  a.P = (int)(npts < prm.op.maxpttrack ? npts : prm.op.maxpttrack);
  a.E = (long long)a.P * prm.op.novals;
  return prm.eigen_packet == 8 ? track_big<16>(a, st) : track_big<8>(a, st);
}

}  // namespace ict
