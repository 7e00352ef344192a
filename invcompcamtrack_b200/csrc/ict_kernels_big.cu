// ict_kernels_big.cu — (1) the multi-CTA form of SetPose + TrackPose for ONE track that is too large for a CTA's
// shared memory (dense full-frame alignment: psz = 1, one point per pixel, BASELINE config 4), and (2) the NCC
// hypothesis scoring kernel.
//
// Same arithmetic as k_track (ict_kernels.cu), including the optional reference-order sums (sum_mode 1: Hessian and
// J^T r by one CTA running Eigen's eight sequential chains, sixteen with 8-float packets); the template (pat_ref, pat_dx, pat_dy) and the per-point state
// live in a global work buffer that fits the 126 MB L2 for a 1080p frame, reductions are two-stage with a fixed
// order (thread-strided partials -> warp tree -> CTA partial -> one finishing CTA), and the iteration loop is a
// fixed sequence of launches whose kernels return immediately once the on-device convergence flag drops, so
// there is still no host round-trip inside TrackPose.
#include "ict_kernels.cuh"
#include "ict_device.cuh"


namespace ict {

int64_t launch_count(int reset);

struct BigState {
  float G[12];
  float p[6];
  Lu6 lu;
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

static inline size_t al(size_t x) { return (x + 255) & ~(size_t)255; }

#define BIG_CHUNK 2048         /* chain elements per staged chunk (8 KB per chain, 64 KB per stage) of the reference-order
                                  chain kernel: every chunk costs ~150 cycles of hand-over on the critical path, so few and
                                  large ones (512 x 4 stages: 0.66 ms per pass of 247 k additions; 2048 x 2: 0.585 ms) */
#define BIG_STAGES 2
// A stage holds 8 * BIG_CHUNK floats whatever the chain count: sixteen chains (8-float packets) take chunks of half the
// length, and their chains are half as long, so the hand-overs per chain pass stay the same.
__host__ __device__ constexpr int big_chunk(int nch) { return 8 * BIG_CHUNK / nch; }
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

size_t bigtrack_work_bytes(const ict_optparam& op, int64_t npts, int eigen_packet) {
  const int64_t P = npts < op.maxpttrack ? npts : op.maxpttrack;
  const int64_t E = P * op.novals;
  size_t b = al(sizeof(BigState));
  b += 4 * al(sizeof(float) * E);
  b += al(sizeof(float) * 10 * P) + al(sizeof(float) * 4 * P) + 4 * al(sizeof(float) * P);
  b += 2 * al(sizeof(int) * P);
  b += al(sizeof(float) * 21 * big_ncta(E));
  const int nch = eigen_packet == 8 ? 16 : 8;
  b += al(sizeof(float) * nch * 24 * (size_t)big_cstride((int64_t)op.maxpttrack * op.novals, nch));   // 24 product rows: the 21 Hessian sums at once
  return b;
}

static BigWork carve(const ict_optparam& op, int64_t npts, int eigen_packet, void* work) {
  const int64_t P = npts < op.maxpttrack ? npts : op.maxpttrack;
  const int64_t E = P * op.novals;
  char* c = (char*)work;
  BigWork w;
  w.st = (BigState*)c; c += al(sizeof(BigState));
  w.ref = (float*)c; c += al(sizeof(float) * E);
  w.gx = (float*)c; c += al(sizeof(float) * E);
  w.gy = (float*)c; c += al(sizeof(float) * E);
  w.pnew = (float*)c; c += al(sizeof(float) * E);
  w.coef = (float*)c; c += al(sizeof(float) * 10 * P);
  w.w = (float*)c; c += al(sizeof(float) * 4 * P);
  w.mean = (float*)c; c += al(sizeof(float) * P);
  w.Xc = (float*)c; c += al(sizeof(float) * P);
  w.Yc = (float*)c; c += al(sizeof(float) * P);
  w.Zc = (float*)c; c += al(sizeof(float) * P);
  w.base = (int*)c; c += al(sizeof(int) * P);
  w.vis = (int*)c; c += al(sizeof(int) * P);
  w.part = (float*)c; c += al(sizeof(float) * 21 * big_ncta(E));
  w.prod = (float*)c;
  w.cstride = big_cstride((int64_t)op.maxpttrack * op.novals, eigen_packet == 8 ? 16 : 8);
  w.ncta = big_ncta(E);
  return w;
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
    track_setpose(a.prm.p_in, a.prm.norm, a.t, op.donorm != 0, S->p, S->G);
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
    save_rotated_point(a.prm, S->G, off, a.n_in, i, q[i], q[a.n_in + i], q[2 * (int64_t)a.n_in + i], a.w.Xc, a.w.Yc,
                       a.w.Zc);
}

__global__ void k_big_level_points(const BigArgs a, int sl) {
  const CamLevels& cam = a.prm.cam;
  const float fx = cam.fx[sl], fy = cam.fy[sl], cx = cam.cx[sl], cy = cam.cy[sl], swo = cam.swo[sl], sho = cam.sho[sl];
  const int width = cam.width[sl];
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.P; i += (long long)gridDim.x * blockDim.x) {
    const float xc = a.w.Xc[i], yc = a.w.Yc[i], zc = a.w.Zc[i];
    const float mx = (xc / zc) * fx + cx;
    const float my = (yc / zc) * fy + cy;
    const bool out = !((mx >= 0) & (my >= 0) & (mx <= swo) & (my <= sho));
    if (out) {
      a.w.vis[i] = 0;
    } else {
      a.w.vis[i] = 1;
      const PatchPlace q = patch_place(mx, my, a.prm.op.pszd2, width);
      a.w.base[i] = q.base;
      a.w.w[i] = q.w0; a.w.w[a.P + i] = q.w1; a.w.w[2LL * a.P + i] = q.w2; a.w.w[3LL * a.P + i] = q.w3;
      float c[10];
      sd_coefs(xc, yc, zc, fx, fy, c);
      for (int k = 0; k < 10; ++k) a.w.coef[(long long)k * a.P + i] = c[k];
    }
  }
}

__global__ void __launch_bounds__(256) k_big_level_gather(const BigArgs a, int sl) {
  const int n = a.prm.op.novals, psz = a.prm.op.psz, width = a.prm.cam.width[sl];
  const int rf = a.prm.fixed_ref;
  const float* __restrict__ Iref = a.prm.frames[rf].I[sl];
  const float* __restrict__ Dxr = a.prm.frames[rf].dx[sl];
  const float* __restrict__ Dyr = a.prm.frames[rf].dy[sl];
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < a.E; e += (long long)gridDim.x * blockDim.x) {
    const long long i = e / n;
    const int rem = (int)(e - i * n), r = rem / psz, c = rem - r * psz;
    if (a.w.vis[i] & 1) {
      const int addr = a.w.base[i] + r * width + c;
      const float w0 = a.w.w[i], w1 = a.w.w[a.P + i], w2 = a.w.w[2LL * a.P + i], w3 = a.w.w[3LL * a.P + i];
      a.w.ref[e] = bilin4(Iref, addr, width, w0, w1, w2, w3);
      a.w.gx[e] = bilin4(Dxr, addr, width, w0, w1, w2, w3);
      a.w.gy[e] = bilin4(Dyr, addr, width, w0, w1, w2, w3);
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
    const long long i = e / n;
    float cf[10], sd[6];
#pragma unroll
    for (int k = 0; k < 10; ++k) cf[k] = a.w.coef[(long long)k * a.P + i];
    sd_values(a.w.gx[e], a.w.gy[e], cf, sd);
    int k = 0;
#pragma unroll
    for (int p = 0; p < 6; ++p)
#pragma unroll
      for (int q = p; q < 6; ++q) { acc[k] = acc[k] + sd[p] * sd[q]; ++k; }
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
  if (threadIdx.x < 32) lu6_factor_warp(s_H, a.w.st->lu);
  if (threadIdx.x == 0) {
    BigState* S = a.w.st;
    const ict_optparam& op = a.prm.op;
    S->normdp_init = 1e-10f;
    S->normdp = 1e-10f;
    S->it = 0;
    S->nvis = 0;
    S->cont = keep_iterating(op, 0, 1e-10f, 1e-10f);
    store_level_iters(a.prm.iters, op, a.t, sl, 0);
  }
}

__global__ void k_big_iter_points(const BigArgs a, int sl) {
  BigState* S = a.w.st;
  if (!S->cont) return;
  const CamLevels& cam = a.prm.cam;
  const float fx = cam.fx[sl], fy = cam.fy[sl], cx = cam.cx[sl], cy = cam.cy[sl], swo = cam.swo[sl], sho = cam.sho[sl];
  const int width = cam.width[sl];
  const int64_t off = a.prm.pt_off[a.t];
  const float* q = a.prm.pt3d + 3 * off;
  int cnt = 0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < a.P; i += (long long)gridDim.x * blockDim.x) {
    float tx, ty, tz;
    rigid_apply<float>(S->G, q[i], q[a.n_in + i], q[2 * (int64_t)a.n_in + i], tx, ty, tz);
    const float mx = (tx / tz) * fx + cx;
    const float my = (ty / tz) * fy + cy;
    const bool out = !((mx >= 0) & (my >= 0) & (mx <= swo) & (my <= sho));
    if (out) {
      a.w.vis[i] &= ~2;
    } else {
      a.w.vis[i] |= 2;
      const PatchPlace pp = patch_place(mx, my, a.prm.op.pszd2, width);
      a.w.base[i] = pp.base;
      a.w.w[i] = pp.w0; a.w.w[a.P + i] = pp.w1; a.w.w[2LL * a.P + i] = pp.w2; a.w.w[3LL * a.P + i] = pp.w3;
      ++cnt;
    }
  }
  // integer count: order-independent
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_down_sync(0xffffffffu, cnt, o);
  if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(&S->nvis, cnt);
}

__global__ void __launch_bounds__(256) k_big_iter_sample(const BigArgs a, int sl) {
  if (!a.w.st->cont) return;
  const int n = a.prm.op.novals, psz = a.prm.op.psz, width = a.prm.cam.width[sl];
  const float* __restrict__ Inew = a.prm.frames[a.prm.fixed_new].I[sl];
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < a.E; e += (long long)gridDim.x * blockDim.x) {
    const long long i = e / n;
    const int rem = (int)(e - i * n), r = rem / psz, c = rem - r * psz;
    if (a.w.vis[i] & 2)
      a.w.pnew[e] = bilin4(Inew, a.w.base[i] + r * width + c, width, a.w.w[i], a.w.w[a.P + i], a.w.w[2LL * a.P + i],
                           a.w.w[3LL * a.P + i]);
  }
}

template <bool PN>
__global__ void __launch_bounds__(256) k_big_iter_elems(const BigArgs a, int sl) {
  if (!a.w.st->cont) return;
  const int n = a.prm.op.novals, psz = a.prm.op.psz, width = a.prm.cam.width[sl];
  const float* __restrict__ Inew = a.prm.frames[a.prm.fixed_new].I[sl];
  float acc[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) acc[k] = 0.0f;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < a.E; e += (long long)gridDim.x * blockDim.x) {
    const long long i = e / n;
    if (a.w.vis[i] & 2) {
      float pn;
      if (PN) {
        pn = a.w.pnew[e];   // mean already subtracted by k_big_patch_means
      } else {
        const int rem = (int)(e - i * n), r = rem / psz, c = rem - r * psz;
        pn = bilin4(Inew, a.w.base[i] + r * width + c, width, a.w.w[i], a.w.w[a.P + i], a.w.w[2LL * a.P + i],
                    a.w.w[3LL * a.P + i]);
      }
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

// solve, pose update, stop rule and trace record of one iteration (one thread); sum6 = the six sums of J^T r
__device__ __forceinline__ void big_iter_finish_serial(const BigArgs& a, int sl, const float* sum6) {
  BigState* S = a.w.st;
  const ict_optparam& op = a.prm.op;
  float sumsd[6], dp[6];
  for (int k = 0; k < 6; ++k) sumsd[k] = sum6[k];
  lu6_solve(S->lu, sumsd, dp);
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
  S->cont = keep_iterating(op, S->it, S->normdp, S->normdp_init);
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
  const float* cf = a.w.coef;
  for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j < nj; j += (long long)gridDim.x * blockDim.x) {
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
      const long long e = NCH * j + c;
      float v[6];
      if (e < lim) {
        const long long i = n == 1 ? e : e / n;
        const float gx = a.w.gx[e], gy = a.w.gy[e];
        float sd[6];
        sd[0] = gx * cf[0 * (long long)a.P + i];
        sd[1] = gy * cf[1 * (long long)a.P + i];
        sd[2] = gx * cf[2 * (long long)a.P + i] + gy * cf[3 * (long long)a.P + i];
        sd[3] = gx * cf[4 * (long long)a.P + i] + gy * cf[5 * (long long)a.P + i];
        sd[4] = gx * cf[6 * (long long)a.P + i] + gy * cf[7 * (long long)a.P + i];
        sd[5] = gx * cf[8 * (long long)a.P + i] + gy * cf[9 * (long long)a.P + i];
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
  const CamLevels& cam = a.prm.cam;
  const float fx = cam.fx[sl], fy = cam.fy[sl], cx = cam.cx[sl], cy = cam.cy[sl], swo = cam.swo[sl], sho = cam.sho[sl];
  const int width = cam.width[sl], n = a.prm.op.novals, psz = a.prm.op.psz, pszd2 = a.prm.op.pszd2;
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
        const float mx = (tx / tz) * fx + cx;
        const float my = (ty / tz) * fy + cy;
        const bool vis = (mx >= 0) & (my >= 0) & (mx <= swo) & (my <= sho);
        float pd = 0.0f;
        if (vis) {
          const PatchPlace pp = patch_place(mx, my, pszd2, width);
          const float pn = bilin4(Inew, pp.base + r * width + cc, width, pp.w0, pp.w1, pp.w2, pp.w3);
          pd = a.w.ref[e] - pn;
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
  constexpr int RS = NCH == 8 ? CH : CH + 4;             // row stride of a stage in shared memory
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

// factorisation + state of a level after the 21 reference-order Hessian sums (part[0..20]) are in
__global__ void __launch_bounds__(32) k_big_hessian_exact_finish(const BigArgs a) {
  __shared__ float s_H[21];
  const int tid = threadIdx.x;
  if (tid < 21) s_H[tid] = a.w.part[tid];
  __syncwarp();
  lu6_factor_warp(s_H, a.w.st->lu);
  if (tid == 0) {
    BigState* S = a.w.st;
    const ict_optparam& op = a.prm.op;
    S->normdp_init = 1e-10f;
    S->normdp = 1e-10f;
    S->it = 0;
    S->nvis = 0;
    S->cont = keep_iterating(op, 0, 1e-10f, 1e-10f);
  }
}

// pdiff of every slot into w.pnew (0 where the point is not visible in the new frame)
template <bool PN>
__global__ void __launch_bounds__(256) k_big_iter_pdiff(const BigArgs a, int sl) {
  if (!a.w.st->cont) return;
  const int n = a.prm.op.novals, psz = a.prm.op.psz, width = a.prm.cam.width[sl];
  const float* __restrict__ Inew = a.prm.frames[a.prm.fixed_new].I[sl];
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < a.E; e += (long long)gridDim.x * blockDim.x) {
    const long long i = e / n;
    float pd = 0.0f;
    if (a.w.vis[i] & 2) {
      float pn;
      if (PN) {
        pn = a.w.pnew[e];
      } else {
        const int rem = (int)(e - i * n), r = rem / psz, c = rem - r * psz;
        pn = bilin4(Inew, a.w.base[i] + r * width + c, width, a.w.w[i], a.w.w[a.P + i], a.w.w[2LL * a.P + i],
                    a.w.w[3LL * a.P + i]);
      }
      pd = a.w.ref[e] - pn;
    }
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
  const CamLevels& cam = a.prm.cam;
  const float fx = cam.fx[sl], fy = cam.fy[sl], cx = cam.cx[sl], cy = cam.cy[sl], swo = cam.swo[sl], sho = cam.sho[sl];
  const int width = cam.width[sl];
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
    const float mx = (xc / zc) * fx + cx;
    const float my = (yc / zc) * fy + cy;
    const bool out = !((mx >= 0) & (my >= 0) & (mx <= swo) & (my <= sho));   // odometer.cpp:273-275
    float sd[6];
    if (!out) {
      const PatchPlace q = patch_place(mx, my, a.prm.op.pszd2, width);      // util_getPatch_grad, one pixel
      a.w.ref[i] = bilin4(Iref, q.base, width, q.w0, q.w1, q.w2, q.w3);
      const float gx = bilin4(Dxr, q.base, width, q.w0, q.w1, q.w2, q.w3);
      const float gy = bilin4(Dyr, q.base, width, q.w0, q.w1, q.w2, q.w3);
      float c[10];
      sd_coefs(xc, yc, zc, fx, fy, c);
      sd_values(gx, gy, c, sd);                                              // odometer.cpp:317-326
#pragma unroll
      for (int k = 0; k < 6; ++k) sdp[k * P + i] = sd[k];
    } else {                               // out of the reference image: the previous level's values stay (SURVEY §9.6)
#pragma unroll
      for (int k = 0; k < 6; ++k) sd[k] = sdp[k * P + i];
    }
    int k = 0;
#pragma unroll
    for (int p = 0; p < 6; ++p)
#pragma unroll
      for (int q = p; q < 6; ++q) { acc[k] = acc[k] + sd[p] * sd[q]; ++k; }
  }
  cta_partials<21>(acc, a.w.part);
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
  const CamLevels& cam = a.prm.cam;
  const float fx = cam.fx[sl], fy = cam.fy[sl], cx = cam.cx[sl], cy = cam.cy[sl], swo = cam.swo[sl], sho = cam.sho[sl];
  const int width = cam.width[sl];
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
  auto sample = [&](long long i, float X, float Y, float Z, bool& vis) -> float {
    float tx, ty, tz;
    rigid_apply(G, X, Y, Z, tx, ty, tz);                                         // project_pt, pose.cpp:307-397
    const float mx = (tx / tz) * fx + cx;
    const float my = (ty / tz) * fy + cy;
    vis = (mx >= 0) & (my >= 0) & (mx <= swo) & (my <= sho);                   // odometer.cpp:369-371
    if (!vis) return 0.0f;
    const PatchPlace pp = patch_place(mx, my, a.prm.op.pszd2, width);
    return bilin4(Inew, pp.base, width, pp.w0, pp.w1, pp.w2, pp.w3);
  };
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
    const float pn0 = sample(i, X0, Y0, Z0, v0);
    const float pn1 = hj ? sample(j, X1, Y1, Z1, v1) : 0.0f;
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
  const CamLevels& cam = a.prm.cam;
  const float fx = cam.fx[sl], fy = cam.fy[sl], cx = cam.cx[sl], cy = cam.cy[sl], swo = cam.swo[sl], sho = cam.sho[sl];
  const int width = cam.width[sl];
  const float* __restrict__ Inew = a.prm.frames[a.prm.fixed_new].I[sl];
  float acc[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) acc[k] = 0.0f;
  int cnt = 0;
  // one point of a staged tile: projection, placement, the four-texel gather (returns the sample, sets vis).
  // (Tried: placing tile n+1 and issuing its gather before folding tile n — 23.1 instead of 21.3 us per iteration.)
  auto sample = [&](int st, bool& vis) -> float {
    const float X = s_buf[st][0][tid], Y = s_buf[st][1][tid], Z = s_buf[st][2][tid];
    float tx, ty, tz;
    rigid_apply(G, X, Y, Z, tx, ty, tz);                                         // project_pt, pose.cpp:307-397
    const float mx = (tx / tz) * fx + cx;
    const float my = (ty / tz) * fy + cy;
    vis = (mx >= 0) & (my >= 0) & (mx <= swo) & (my <= sho);                   // odometer.cpp:369-371
    if (!vis) return 0.0f;
    const PatchPlace pp = patch_place(mx, my, a.prm.op.pszd2, width);
    return bilin4(Inew, pp.base, width, pp.w0, pp.w1, pp.w2, pp.w3);
  };
  for (int n = 0; n < nmine; ++n) {
    const int st = n % NST;
    const long long i = ((long long)blockIdx.x + (long long)n * gridDim.x) * 256 + tid;
    mbar_wait(&s_full[st], (n / NST) & 1);
    bool vis = false;
    float pn = 0.0f;
    if (i < P) pn = sample(st, vis);
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

__global__ void k_big_level_end(const BigArgs a, int sl) {
  store_level_iters(a.prm.iters, a.prm.op, a.t, sl, a.w.st->it);
}

__global__ void k_big_final(const BigArgs a) {
  const BigState* S = a.w.st;
  finish_track(a.prm, a.t, a.prm.op.donorm != 0, S->p, S->G, a.prm.p_out, a.prm.npixres, S->npix,
               track_trace(a.prm, a.t), S->trace_n);
}

cudaError_t launch_track_big(const TrackParams& prm, int t, int64_t npts, void* work, cudaStream_t st) {
  BigArgs a;
  a.prm = prm;
  a.w = carve(prm.op, npts, prm.eigen_packet, work);
  a.t = t;
  a.n_in = (int)npts;
  a.P = (int)(npts < prm.op.maxpttrack ? npts : prm.op.maxpttrack);
  a.E = (long long)a.P * prm.op.novals;
  const ict_optparam& op = prm.op;
  const int ncta = a.w.ncta;
  const int pcta_ = (int)((a.P + 255) / 256 < 148 * 8 ? (a.P + 255) / 256 : 148 * 8);
  const int pcta = pcta_ > 0 ? pcta_ : 1;   // an empty track still runs the launch chain (its sums are empty, its pose unchanged)
  const bool pn = op.dopatchnorm != 0;
  const bool ex = prm.sum_mode != 0;   // reference-order sums
  const bool pk8 = ex && prm.eigen_packet == 8;   // ... with 8-float packets: sixteen chains per sum
  const bool fused = !pn && !ex && !prm.force_general && op.novals == 1;
  int nl = 0;
  const size_t chain_smem = pk8 ? sizeof(float) * BIG_STAGES * 16 * (big_chunk(16) + 4)    // 128.5 KB
                                : sizeof(float) * BIG_STAGES * 8 * BIG_CHUNK;                  // 128 KB
  if (ex) {
    const cudaError_t e = pk8 ? set_kernel_attrs<k_big_chains<16>>((int)chain_smem, -1)
                              : set_kernel_attrs<k_big_chains<8>>((int)chain_smem, -1);
    if (e != cudaSuccess) return e;
  }
  k_big_init<<<ncta, 256, 0, st>>>(a, fused ? 1 : 0); ++nl;
  k_big_project_ref<<<pcta, 256, 0, st>>>(a); ++nl;
  for (int sl = op.lv_f; sl >= op.lv_l && fused; --sl) {   // dense path: one launch per level + one per iteration
    // bulk-copy staging needs 16-byte aligned streams: point counts and the track's offset multiples of four
    const bool tma = t == 0 && (a.P % 4 == 0) && (a.n_in % 4 == 0);   // t == 0: offset 0
    // programmatic dependent launch: iteration k+1 becomes resident while the last CTA of iteration k still runs the
    // solve, and its first tiles are in flight by the time the pose is published
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute lattr[1];
    lattr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    lattr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.gridDim = dim3(ncta);
    cfg.blockDim = dim3(256);
    cfg.stream = st;
    cfg.attrs = lattr;
    cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, k_dense_level, a, sl); ++nl;
    cfg.gridDim = dim3(1);
    cudaLaunchKernelEx(&cfg, k_big_level_finish, a, sl); ++nl;
    cfg.gridDim = dim3(ncta);
    for (int it = 0; it < op.maxiter; ++it) {
      if (tma) { cfg.dynamicSmemBytes = 3 * 10240; cudaLaunchKernelEx(&cfg, k_dense_iter_tma<3>, a, sl); }
      else k_dense_iter<<<ncta, 256, 0, st>>>(a, sl);
      ++nl;
    }
    // (no k_big_level_end: the iteration's serial tail records the level's iteration count)
  }
  for (int sl = op.lv_f; sl >= op.lv_l && !fused; --sl) {
    k_big_level_points<<<pcta, 256, 0, st>>>(a, sl); ++nl;
    k_big_level_gather<<<ncta, 256, 0, st>>>(a, sl); ++nl;
    if (pn) { k_big_patch_means<<<pcta, 256, 0, st>>>(a, a.w.ref, 1, 1, ex ? prm.eigen_packet : 0); ++nl; }
    if (ex) {
      // the products of all 21 sums (four passes of six rows), then their 21 x 8 chains side by side: one chain pass
      // (E / 8 dependent additions) per level instead of four
      for (int pass = 0; pass < 4; ++pass) {
        if (pk8) k_big_products<1, 16><<<ncta, 256, 0, st>>>(a, pass); else k_big_products<1, 8><<<ncta, 256, 0, st>>>(a, pass);
        ++nl;
      }
      if (pk8) k_big_chains<16><<<21, 64, chain_smem, st>>>(a, 21, a.w.part, 0); else k_big_chains<8><<<21, 64, chain_smem, st>>>(a, 21, a.w.part, 0);
      ++nl;
      k_big_hessian_exact_finish<<<1, 32, 0, st>>>(a); ++nl;
    } else {
      k_big_level_hessian<<<ncta, 256, 0, st>>>(a); ++nl;
      k_big_level_finish<<<1, 256, 0, st>>>(a, sl); ++nl;
    }
    for (int it = 0; it < op.maxiter; ++it) {
      if (ex && !pn && a.E <= (1 << 18)) {
        // three launches per iteration instead of five: products of all elements, the chains, the serial tail.  For
        // tracks whose launches are latency-bound; beyond ~256 k elements the three streaming kernels below are faster
        // than the fused one.  (The serial tail inside the chain kernel's last CTA was measured: passing the argument
        // block on costs the chain kernel a local copy of it, 26 -> 32 ms per dense TrackPose.)
        if (pk8) {
          k_big_iter_fused_exact<16><<<ncta, 256, 0, st>>>(a, sl);
          k_big_chains<16><<<6, 64, chain_smem, st>>>(a, 6, a.w.part, 1);
        } else {
          k_big_iter_fused_exact<8><<<ncta, 256, 0, st>>>(a, sl);
          k_big_chains<8><<<6, 64, chain_smem, st>>>(a, 6, a.w.part, 1);
        }
        nl += 2;
        k_big_iter_finish<<<1, 256, 0, st>>>(a, sl, 1); ++nl;
        continue;
      }
      k_big_iter_points<<<pcta, 256, 0, st>>>(a, sl); ++nl;
      if (pn) {
        k_big_iter_sample<<<ncta, 256, 0, st>>>(a, sl); ++nl;
        k_big_patch_means<<<pcta, 256, 0, st>>>(a, a.w.pnew, 2, 1, ex ? prm.eigen_packet : 0); ++nl;
      }
      if (ex) {
        if (pn) k_big_iter_pdiff<true><<<ncta, 256, 0, st>>>(a, sl); else k_big_iter_pdiff<false><<<ncta, 256, 0, st>>>(a, sl);
        ++nl;
        if (pk8) {
          k_big_products<0, 16><<<ncta, 256, 0, st>>>(a, 0);
          k_big_chains<16><<<6, 64, chain_smem, st>>>(a, 6, a.w.part, 1);
        } else {
          k_big_products<0, 8><<<ncta, 256, 0, st>>>(a, 0);
          k_big_chains<8><<<6, 64, chain_smem, st>>>(a, 6, a.w.part, 1);
        }
        nl += 2;
      } else {
        if (pn) k_big_iter_elems<true><<<ncta, 256, 0, st>>>(a, sl); else k_big_iter_elems<false><<<ncta, 256, 0, st>>>(a, sl);
        ++nl;
      }
      k_big_iter_finish<<<1, 256, 0, st>>>(a, sl, ex ? 1 : ncta); ++nl;
    }
    k_big_level_end<<<1, 1, 0, st>>>(a, sl); ++nl;
  }
  k_big_final<<<1, 1, 0, st>>>(a); ++nl;
  for (int k = 0; k < nl; ++k) count_launch();
  return cudaGetLastError();
}

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
