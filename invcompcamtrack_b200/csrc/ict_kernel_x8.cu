// ict_kernel_x8.cu — K2x8: SetPose + TrackPose for 8x8 patches with the REFERENCE'S ORDER OF SUMMATION
// (ict_tracker_set_sum_order(tr, 1)), with or without dopatchnorm: bit-identical to the oracle's default model of
// the reference like k_track<8, 2|3> (ict_kernels.cu), organised like K2x (ict_kernel_x.cu) so that the sequential
// chains do not leave the CTA idle — the reference's own configuration (psz 8, ~100 points per track) ran at 14 ms
// per TrackPose in that mode with one thread per chain.
//
// With e = point*64 + row*8 + col, chain c of Eigen's packet sum IS column c: it adds rows 0..7 of point 0, then of
// point 1, ...  A tile is one patch.  Producer warp w makes the patches 7j + w (round j): lane l takes the pixels
// (2q, c) and (2q+1, c), q = l/8, c = l%8 (the K2v8 lane layout), computes the six values to be summed of both
// pixels with the reference's roundings and stores them as stage[k][c][row]; the chain warp's lane (k, c) reads its
// column with two LDS.128 and performs the eight additions of the patch in row order.  Ring halves of seven
// patches are handed over with mbarriers as in K2x.  Every producer computes the placement of ITS patches with
// lanes = patches after the iteration barrier, so the chain warp — the critical resource — only combines the chains,
// solves (Eigen's elimination, straight-line, true divisions) and evaluates the reference's exp.
//
// dopatchnorm in the reference order: the mean of a patch is Eigen's sum of its 64 values, i.e. the same eight
// column chains followed by the redux tail; a patch lives in one warp, so the chain of column c runs through the four
// lanes that hold its rows (three shuffles) and the tail through the last row group's lanes.
//
// With Eigen's 8-float packets (sum order 3, PK = 8) a sum has sixteen chains: chain c adds e = c, c + 16, ...  For 8x8
// patches that is chain (row & 1) * 8 + col, four rows of one parity per patch; for 16x16 patches chain c is column
// c.  In both cases a staged column of eight values holds two chains, the even positions and the odd ones, so the
// chain lane (k, c) keeps two accumulators per quantity, each half as long, and adds them (p0 + p1) before the tail.
#include "ict_kernels.cuh"
#include "ict_device.cuh"
#include "ict_kernel_v2.cuh"
#include "ict_kernel_v8.cuh"
#include "ict_kernel_x.cuh"

namespace ict {


#define X8_TILE 384                     /* floats per staged patch: six quantities x 8 columns x 8 rows */
#define X8_MAXR 32                      /* rounds per sum at most: 7 * 32 = 224 points per track */

// Eigen's vectorised sum of the 64 values of a patch held two per lane (rows 2q, 2q+1 of column c; lane = 8q + c):
// PK = 4: chain c = ((((v[0][c] + v[1][c]) + v[2][c]) + ...) + v[7][c]), then (c0+c4 + c2+c6) + (c1+c5 + c3+c7).
// PK = 8: chains (even rows of c) and (odd rows of c), their sum per column, then the same tail.
// Returns the sum in every lane.
template <int PK>
__device__ __forceinline__ float x8_patch_sum(float a, float b) {
  const unsigned FULL = 0xffffffffu;
  const int q = (threadIdx.x & 31) >> 3;
  float s;
  if (PK == 4) {
    s = a + b;                                            // rows 0, 1 (valid in row group 0)
#pragma unroll
    for (int step = 1; step < 4; ++step) {
      const float t = __shfl_up_sync(FULL, s, 8);
      if (q == step) s = (t + a) + b;
    }
  } else {
    float se = a, so = b;                                 // rows 0 and 1 (valid in row group 0)
#pragma unroll
    for (int step = 1; step < 4; ++step) {
      const float te = __shfl_up_sync(FULL, se, 8), to = __shfl_up_sync(FULL, so, 8);
      if (q == step) { se = te + a; so = to + b; }
    }
    s = se + so;                                          // p0[c] + p1[c]
  }
  // lanes 24..31 hold the chains of columns 0..7
  const float p0 = s + __shfl_down_sync(FULL, s, 4);      // lanes 24..27: ch[c] + ch[c+4]
  const float t2 = p0 + __shfl_down_sync(FULL, p0, 2);    // lane 24: p0[0] + p0[2]; lane 25: p0[1] + p0[3]
  const float r = t2 + __shfl_down_sync(FULL, t2, 1);     // lane 24
  return __shfl_sync(FULL, r, 24);
}

// chain warp, one round of staged patches: chain (k, c) adds rows 0..7 of column c, patch after patch.  The quads of
// patch w + 1 are loaded before the sixteen dependent additions of patch w, so that their latency (and the shared-
// memory pipe's four cycles per LDS.128) is covered by the additions instead of preceding them.
struct X8Quads {
  float4 x0, x1, y0, y1;
};
__device__ __forceinline__ void x8_load(const float* tile, int lane, X8Quads& q) {
  const int c = lane & 7, kx = lane >> 3;
  const float4* px = reinterpret_cast<const float4*>(tile + (kx * 8 + c) * 8);
  const float4* py = reinterpret_cast<const float4*>(tile + ((4 + kx) * 8 + c) * 8);
  // a column's eight rows are 32 bytes: columns c and c + 4 share their banks, so columns 4..7 keep their two row
  // quads swapped (x8_store) — the eight lanes of an LDS.128 phase then cover all 32 banks
  const int lo = (c >> 2) & 1;
  q.x0 = px[lo];
  q.x1 = px[lo ^ 1];
  q.y0 = q.y1 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (lane < 16) { q.y0 = py[lo]; q.y1 = py[lo ^ 1]; }
}
// s[0], s[1]: the chains of quantities kx and 4 + kx; with PK = 8 these take the even positions of the column and
// s[2], s[3] the odd ones
template <int PK>
__device__ __forceinline__ void x8_add(const X8Quads& q, bool first, float* s) {
  if (PK == 4) {
    float sx = s[0], sy = s[1];
    sx = first ? q.x0.x : sx + q.x0.x;  sy = first ? q.y0.x : sy + q.y0.x;
    sx = sx + q.x0.y; sy = sy + q.y0.y; sx = sx + q.x0.z; sy = sy + q.y0.z; sx = sx + q.x0.w; sy = sy + q.y0.w;
    sx = sx + q.x1.x; sy = sy + q.y1.x; sx = sx + q.x1.y; sy = sy + q.y1.y; sx = sx + q.x1.z; sy = sy + q.y1.z; sx = sx + q.x1.w; sy = sy + q.y1.w;
    s[0] = sx; s[1] = sy;
  } else {
    float xe = s[0], ye = s[1], xo = s[2], yo = s[3];
    xe = first ? q.x0.x : xe + q.x0.x;  ye = first ? q.y0.x : ye + q.y0.x;
    xo = first ? q.x0.y : xo + q.x0.y;  yo = first ? q.y0.y : yo + q.y0.y;
    xe = xe + q.x0.z; ye = ye + q.y0.z; xo = xo + q.x0.w; yo = yo + q.y0.w;
    xe = xe + q.x1.x; ye = ye + q.y1.x; xo = xo + q.x1.y; yo = yo + q.y1.y;
    xe = xe + q.x1.z; ye = ye + q.y1.z; xo = xo + q.x1.w; yo = yo + q.y1.w;
    s[0] = xe; s[1] = ye; s[2] = xo; s[3] = yo;
  }
}
// the two quantities' chains, combined per lane: the chain of column c (PK = 4) or p0[c] + p1[c] (PK = 8)
template <int PK>
__device__ __forceinline__ float2 x8_lane_chains(const float* s) {
  return PK == 4 ? make_float2(s[0], s[1]) : make_float2(s[0] + s[2], s[1] + s[3]);
}
template <int NP, int PK>
__device__ __forceinline__ void x8_consume_round(const float* half, int lane, int j, int ntile, float* s) {
  X8Quads cur, nxt;
  x8_load(half, lane, cur);
  if ((j + 1) * NP <= ntile) {
#pragma unroll
    for (int w = 0; w < NP; ++w) {
      if (w + 1 < NP) x8_load(half + (w + 1) * X8_TILE, lane, nxt);
      x8_add<PK>(cur, w == 0 && j == 0, s);
      cur = nxt;
    }
  } else {
    const int n = ntile - j * NP;
    for (int w = 0; w < n; ++w) {
      if (w + 1 < n) x8_load(half + (w + 1) * X8_TILE, lane, nxt);
      x8_add<PK>(cur, w == 0 && j == 0, s);
      cur = nxt;
    }
  }
}

// producer: the six values of the lane's two pixels -> stage[k][c][2q], [2q+1]
__device__ __forceinline__ void x8_store(float* tile, int q, int c, const float* v0, const float* v1) {
#pragma unroll
  for (int k = 0; k < 6; ++k)
    *reinterpret_cast<float2*>(tile + (k * 8 + c) * 8 + ((2 * q) ^ (c & 4))) = make_float2(v0[k], v1[k]);
}

// The lane's texels for its two pixels of a tile.  TPP = tiles per point: 1 for 8x8 patches (a tile = the patch, lane
// (q, c) = rows 2q, 2q + 1 of column c: three texel rows, shared middle one), 4 for 16x16 patches (tile tt = rows 4 tt ..
// 4 tt + 3; with e = row * 16 + col chain c adds (row, c), (row, c + 8) row after row, so lane (q, c) = columns c and
// c + 8 of row 4 tt + q: two texel rows, two column pairs).  Pixel (r, x) of a patch reads the texels at
// base + r * width + x, - 1, - width, - width - 1 (bilin4).
template <int TPP>
struct XRows {
  float v[TPP == 1 ? 6 : 8];
};
template <int TPP>
__device__ __forceinline__ XRows<TPP> x_load(const float* __restrict__ pl, int base, int tt, int q, int c, int width) {
  XRows<TPP> r;
  if (TPP == 1) {
    const int o = base + (2 * q - 1) * width + c;
    r.v[0] = __ldg(pl + o);             r.v[1] = __ldg(pl + o - 1);
    r.v[2] = __ldg(pl + o + width);     r.v[3] = __ldg(pl + o + width - 1);
    r.v[4] = __ldg(pl + o + 2 * width); r.v[5] = __ldg(pl + o + 2 * width - 1);
  } else {
    const int o = base + (4 * tt + q - 1) * width + c;
    r.v[0] = __ldg(pl + o);             r.v[1] = __ldg(pl + o - 1);
    r.v[2] = __ldg(pl + o + width);     r.v[3] = __ldg(pl + o + width - 1);
    r.v[4] = __ldg(pl + o + 8);         r.v[5] = __ldg(pl + o + 7);
    r.v[6] = __ldg(pl + o + width + 8); r.v[7] = __ldg(pl + o + width + 7);
  }
  return r;
}
// util_getPatch / util_getPatch_grad (utilities.cpp:107, 181-183), unfused, reference order: the lane's two pixels
template <int TPP>
__device__ __forceinline__ float2 x_bilin(const XRows<TPP>& r, const float4 w) {
  float2 v;
  v.x = ((w.x * r.v[2] + w.y * r.v[3]) + w.z * r.v[0]) + w.w * r.v[1];
  if (TPP == 1) v.y = ((w.x * r.v[4] + w.y * r.v[5]) + w.z * r.v[2]) + w.w * r.v[3];
  else v.y = ((w.x * r.v[6] + w.y * r.v[7]) + w.z * r.v[4]) + w.w * r.v[5];
  return v;
}

// NP producer warps + the chain warp.  NP = 7: 256 threads, two CTAs per SM up to 100 points per track (throughput form).
// NP = 15: 512 threads, one CTA per SM — a producer's round is ~150 dependent unfused instructions (~900 cycles), so
// the time of an iteration is rounds x 900 and twice the producers halve it; chosen when only one CTA fits an SM anyway
// or when the batch is too small to fill the GPU twice (the reference's own use: one track per call).
template <bool PN, int NP, int TPP, int PK>
__global__ void __launch_bounds__((NP + 1) * 32, NP == 7 ? 2 : 1) k_track_x8(const TrackParams prm) {
  constexpr int N = 64 * TPP;          // pixels per patch
  extern __shared__ __align__(16) float smem[];
  __shared__ KxShared S;
  __shared__ int s_nv[NP + 1];

  const int t = blockIdx.x + prm.t0;
  const ict_optparam& op = prm.op;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int64_t off = prm.pt_off[t];
  const int n_in = (int)(prm.pt_off[t + 1] - off);
  const int P = min(n_in, op.maxpttrack);
  const bool donorm = op.donorm != 0;
  const bool pnorm = PN && op.dopatchnorm != 0;
  const int q2 = lane >> 3, cc = lane & 7;
  const int Q = P * TPP;                  // tiles of the track: 64 pixel-values of every sum each
  const int ROUNDS = (Q + NP - 1) / NP;

  float2* s_ref2 = reinterpret_cast<float2*>(smem);    // [Q][32]: the lane's two pixels of the tile (XRows), lane = 8q + c
  float2* s_gx2 = s_ref2 + 32 * Q;
  float2* s_gy2 = s_gx2 + 32 * Q;
  float* s_ring = reinterpret_cast<float*>(s_gy2 + 32 * Q);   // [2][NP][X8_TILE]
  float4* s_rpl = reinterpret_cast<float4*>(s_ring + 2 * NP * X8_TILE);   // [P][2] reference placement
  float4* s_npl = s_rpl + 2 * P;                        // [P][2] new-frame placement
  float* s_AB = reinterpret_cast<float*>(s_npl + 2 * P);    // [P][12]
  float* s_X = s_AB + 12 * P;
  float* s_Y = s_X + P;
  float* s_Z = s_Y + P;
  float* s_Xc = s_Z + P;
  float* s_Yc = s_Xc + P;
  float* s_Zc = s_Yc + P;

  const TrackFrames fr = track_frames(prm, t);
  const bool chainw = warp == NP;

  // ---- ResetOdometer (odometer.cpp:580-609) + points -----------------------------------------------------------------
  // ResetOdometer runs from the constructor and from Set3Dpoints only (odometer.cpp:153, 173): between the TrackPose
  // calls of one sample (the chains of run_track_nposes.cpp:232-258) the patch and steepest-descent arrays keep their
  // contents, so a point that has left the image keeps the template of the last level it was seen at — also from a
  // PREVIOUS frame step.  With the tracker's "keep_state" the arrays of this CTA (template planes + the per-point sd
  // coefficients they were made with) are therefore carried through global memory from call to call.
  float* state = prm.state ? prm.state + (int64_t)t * prm.state_stride : nullptr;
  {
    const float2 z2 = make_float2(0.f, 0.f);
    const float2* st2 = reinterpret_cast<const float2*>(state);
    const bool load = state && prm.state_load;
    for (int e = tid; e < 3 * 32 * Q; e += nt) s_ref2[e] = load ? st2[e] : z2;
    const float* q = prm.pt3d + 3 * off;
    for (int i = tid; i < P; i += nt) {
      s_X[i] = q[i];
      s_Y[i] = q[n_in + i];
      s_Z[i] = q[2 * (int64_t)n_in + i];
#pragma unroll
      for (int k = 0; k < 12; ++k) s_AB[i * 12 + k] = load ? state[3 * 64 * P + i * 12 + k] : 0.0f;
    }
  }
  if (tid == 0) track_setpose(prm.p_in, prm.norm, t, donorm, S.p, S.G);
  if (tid >= 32 && tid < 34) {
    mbar_init(&S.full[tid - 32], 32 * NP);
    mbar_init(&S.empty[tid - 32], 32);
  }
  __syncthreads();
  for (int i = tid; i < P; i += nt) save_rotated_point(prm, S.G, off, n_in, i, s_X[i], s_Y[i], s_Z[i], s_Xc, s_Yc, s_Zc);
  __syncthreads();

  float* trace = track_trace(prm, t);
  int trace_n = 0;
  float normdp_init = 1e-10f;
  int nvsum = 0;
  int ground = 0;                 // rounds done so far, counted alike by every warp: half = ground & 1, use = ground >> 1

  for (int sl = op.lv_f; sl >= op.lv_l; --sl) {
    const float fx = prm.cam.fx[sl], fy = prm.cam.fy[sl], cx = prm.cam.cx[sl], cy = prm.cam.cy[sl];
    const float swo = prm.cam.swo[sl], sho = prm.cam.sho[sl];
    const int width = prm.cam.width[sl];
    const float* __restrict__ Iref = fr.ref->I[sl];
    const float* __restrict__ Dxr = fr.ref->dx[sl];
    const float* __restrict__ Dyr = fr.ref->dy[sl];
    const float* __restrict__ Inew = fr.nw->I[sl];

    // ---- 4a. per point: reference placement + steepest-descent coefficients (odometer.cpp:268-279, 306-326) ------
    for (int i = tid; i < P; i += nt) {
      const float xc = s_Xc[i], yc = s_Yc[i], zc = s_Zc[i];
      const float mx = (xc / zc) * fx + cx, my = (yc / zc) * fy + cy;
      const int vis = (mx >= 0) & (my >= 0) & (mx <= swo) & (my <= sho);
      PatchPlace pl = {0, 0.f, 0.f, 0.f, 0.f};
      if (vis) {
        pl = patch_place(mx, my, 4 * (TPP == 1 ? 1 : 2), width);
        float c[10];
        sd_coefs(xc, yc, zc, fx, fy, c);
        float* ab = s_AB + i * 12;
        ab[0] = c[0]; ab[1] = 0.0f; ab[2] = c[2]; ab[3] = c[4]; ab[4] = c[6]; ab[5] = c[8];
        ab[6] = 0.0f; ab[7] = c[1]; ab[8] = c[3]; ab[9] = c[5]; ab[10] = c[7]; ab[11] = c[9];
      }
      s_rpl[2 * i] = make_float4(__int_as_float(pl.base), __int_as_float(vis), 0.0f, 0.0f);
      s_rpl[2 * i + 1] = make_float4(pl.w0, pl.w1, pl.w2, pl.w3);
    }
    __syncthreads();
    // ---- 4b. template gather (all eight warps; util_getPatch_grad, unfused, reference order) ------------------------
    for (int i = warp; i < Q; i += NP + 1) {
      const int ip = i / TPP, tt = i % TPP;
      const float4 pa = s_rpl[2 * ip], pw = s_rpl[2 * ip + 1];
      if (__float_as_int(pa.y)) {
        const int o = __float_as_int(pa.x);
        const XRows<TPP> ri = x_load<TPP>(Iref, o, tt, q2, cc, width), rx = x_load<TPP>(Dxr, o, tt, q2, cc, width),
                         ry = x_load<TPP>(Dyr, o, tt, q2, cc, width);
        float2 r = x_bilin<TPP>(ri, pw);
        if (pnorm) {                     // utilities.cpp:187-188: tmp.sum() / novals, Eigen's order
          const float m = x8_patch_sum<PK>(r.x, r.y) / N;
          r.x = r.x - m;
          r.y = r.y - m;
        }
        s_ref2[i * 32 + lane] = r;
        s_gx2[i * 32 + lane] = x_bilin<TPP>(rx, pw);
        s_gy2[i * 32 + lane] = x_bilin<TPP>(ry, pw);
      }
    }
    __syncthreads();

    // ---- 6. Hessian: 21 reference-order sums in four passes of six (odometer.cpp:428-472) --------------------------
#pragma unroll 1
    for (int pass = 0; pass < 4; ++pass) {
      if (!chainw) {
        for (int j = 0; j < ROUNDS; ++j) {
          const int h = ground & 1, use = ground >> 1;
          if (use > 0) mbar_wait_relaxed(&S.empty[h], (use - 1) & 1);
          const int i = j * NP + warp;
          if (i < Q) {
            const float2 GX = s_gx2[i * 32 + lane], GY = s_gy2[i * 32 + lane];
            float ab[12];
#pragma unroll
            for (int k = 0; k < 12; ++k) ab[k] = s_AB[(i / TPP) * 12 + k];
            float sd0[6], sd1[6], v0[6], v1[6];
            kx_sd(GX.x, GY.x, ab, sd0);
            kx_sd(GX.y, GY.y, ab, sd1);
            switch (pass) {
              case 0: kx_hess_products<0>(sd0, v0); kx_hess_products<0>(sd1, v1); break;
              case 1: kx_hess_products<1>(sd0, v0); kx_hess_products<1>(sd1, v1); break;
              case 2: kx_hess_products<2>(sd0, v0); kx_hess_products<2>(sd1, v1); break;
              default: kx_hess_products<3>(sd0, v0); kx_hess_products<3>(sd1, v1); break;
            }
            x8_store(s_ring + (h * NP + warp) * X8_TILE, q2, cc, v0, v1);
          }
          mbar_arrive(&S.full[h]);
          ++ground;
        }
      } else {
        float s4[4] = {0.0f, 0.0f, 0.0f, 0.0f};
        for (int j = 0; j < ROUNDS; ++j) {
          const int h = ground & 1;
          mbar_wait(&S.full[h], (ground >> 1) & 1);
          x8_consume_round<NP, PK>(s_ring + h * NP * X8_TILE, lane, j, Q, s4);
          mbar_arrive(&S.empty[h]);
          ++ground;
        }
        const float2 ch = x8_lane_chains<PK>(s4);
        const float rx = kx_finish(ch.x), ry = kx_finish(ch.y);
        if ((lane & 7) == 0) {
          const int q = 6 * pass + (lane >> 3);
          if (q < 21) S.Hsum[q] = rx;
          if (lane < 16 && q + 4 < 21) S.Hsum[q + 4] = ry;
        }
      }
    }
    // ---- factorisation ---------------------------------------------------------------------------------------------------
    if (chainw) {
      __syncwarp();
      lu6_factor_warp(S.Hsum, S.f);      // Eigen's fullPivLu, bit-identical
      normdp_init = 1e-10f;              // odometer.cpp:341-342
      if (lane == 0) {
        S.it = 0;
        S.cont = keep_iterating(op, 0, 1e-10f, 1e-10f);
      }
    }
    __syncthreads();

    // ---- iterations (odometer.cpp:344-419) ----------------------------------------------------------------------------
    int it = 0;
    while (S.cont) {
      float s4[4] = {0.0f, 0.0f, 0.0f, 0.0f};
      if (!chainw) {
        // 7. project_pt + new-frame placement of this warp's patches (7m + warp), lanes = patches
        {
          const int i = lane * NP + warp;
          int v = 0;
          if (i < P) v = place_point(S.G, s_X[i], s_Y[i], s_Z[i], fx, fy, cx, cy, swo, sho, width, s_npl + 2 * i, 4 * (TPP == 1 ? 1 : 2));
          const int nvw = __popc(__ballot_sync(0xffffffffu, v));
          if (lane == 0) s_nv[warp] = nvw;
        }
        __syncwarp();
        // with several tiles per patch a warp's tiles belong to points placed by other producer warps
        if (TPP > 1) asm volatile("bar.sync 2, %0;" ::"n"(NP * 32) : "memory");
        // 8. one patch per round; the new-frame rows of a patch are fetched TWO rounds ahead: a round is shorter than
        // the L2 round trip of the gather (~900 cycles), so with one round of lead every producer stalled on its loads
        // and the chain warp on the producers
        struct Pre {
          XRows<TPP> ln;
          float4 lw;
          bool lvis;
        };
        auto fetch = [&](int i, Pre& o) {
          const int ip = i / TPP;
          const float4 pa = s_npl[2 * ip];
          o.lw = s_npl[2 * ip + 1];
          o.lvis = __float_as_int(pa.y) != 0;
          if (o.lvis) o.ln = x_load<TPP>(Inew, __float_as_int(pa.x), i % TPP, q2, cc, width);
        };
        Pre cur, nx1, nx2;
#pragma unroll
        for (int k = 0; k < (TPP == 1 ? 6 : 8); ++k) cur.ln.v[k] = 0.0f;
        cur.lw = make_float4(0.f, 0.f, 0.f, 0.f);
        cur.lvis = false;
        nx1 = cur;
        nx2 = cur;
        if (warp < Q) fetch(warp, cur);
        if (warp + NP < Q) fetch(warp + NP, nx1);
        for (int j = 0; j < ROUNDS; ++j) {
          const int i = j * NP + warp;
          const int h = ground & 1, use = ground >> 1;
          const bool have = i < Q;
          float v0[6], v1[6];
          if (i + 2 * NP < Q) fetch(i + 2 * NP, nx2);
          if (have) {
            const bool vis = cur.lvis;
            float2 pn = make_float2(0.f, 0.f);
            if (vis) {
              pn = x_bilin<TPP>(cur.ln, cur.lw);     // util_getPatch (utilities.cpp:55-113), unfused
              if (pnorm) {                           // utilities.cpp:111-112, Eigen's order
                const float mn = x8_patch_sum<PK>(pn.x, pn.y) / N;
                pn.x = pn.x - mn;
                pn.y = pn.y - mn;
              }
            }
            const float2 R = s_ref2[i * 32 + lane], GX = s_gx2[i * 32 + lane], GY = s_gy2[i * 32 + lane];
            float ab[12];
#pragma unroll
            for (int k = 0; k < 12; ++k) ab[k] = s_AB[(i / TPP) * 12 + k];
            float sd0[6], sd1[6];
            kx_sd(GX.x, GY.x, ab, sd0);
            kx_sd(GX.y, GY.y, ab, sd1);
            const float p0 = vis ? R.x - pn.x : 0.0f, p1 = vis ? R.y - pn.y : 0.0f;   // pdiff, odometer.cpp:381
#pragma unroll
            for (int k = 0; k < 6; ++k) { v0[k] = sd0[k] * p0; v1[k] = sd1[k] * p1; }   // sd_k_proj, :386-391
          }
          if (use > 0) mbar_wait_relaxed(&S.empty[h], (use - 1) & 1);
          if (have) x8_store(s_ring + (h * NP + warp) * X8_TILE, q2, cc, v0, v1);
          mbar_arrive(&S.full[h]);
          ++ground;
          cur = nx1;
          nx1 = nx2;
        }
      } else {
        long long tc0 = 0, tw = 0, tcons = 0;   // instrumentation (trace only)
        if (trace) tc0 = clock64();
        for (int j = 0; j < ROUNDS; ++j) {
          const int h = ground & 1;
          if (trace && j == 0) {
            const long long ta = clock64();
            mbar_wait(&S.full[h], (ground >> 1) & 1);
            tw = clock64() - ta;
          } else {
            mbar_wait(&S.full[h], (ground >> 1) & 1);
          }
          const long long tq = trace ? clock64() : 0;
          x8_consume_round<NP, PK>(s_ring + h * NP * X8_TILE, lane, j, Q, s4);
          if (trace) tcons += clock64() - tq;
          mbar_arrive(&S.empty[h]);
          ++ground;
        }
        const long long tc1 = trace ? clock64() : 0;
        // 9a. sumsd[k]: Eigen's redux of the eight (sixteen) chains
        const float2 ch = x8_lane_chains<PK>(s4);
        const float rx = kx_finish(ch.x), ry = kx_finish(ch.y);
        if ((lane & 7) == 0) {
          S.sum[lane >> 3] = rx;
          if (lane < 16) S.sum[4 + (lane >> 3)] = ry;
        }
        __syncwarp();
        int nv = 0;
        if (lane == 0) {
          // s_nv reaches this warp through the ring's barriers; an empty track has no rounds, and no visible point
          if (ROUNDS > 0)
            for (int w = 0; w < NP; ++w) nv += s_nv[w];
          float sumsd[6], dp[6];
#pragma unroll
          for (int k = 0; k < 6; ++k) sumsd[k] = S.sum[k];
          lu6_solve_exact(S.f, S.sum, S.dp);                     // 9b. odometer.cpp:407, Eigen's substitution order
          float pr[6], Gr[12];
#pragma unroll
          for (int k = 0; k < 6; ++k) { dp[k] = S.dp[k]; pr[k] = S.p[k] + dp[k]; S.p[k] = pr[k]; }   // 10. addpose_se3
          Gr[3] = Gr[7] = Gr[11] = 0.0f;
          se3_exp<float>(Gr, pr);
#pragma unroll
          for (int k = 0; k < 12; ++k) S.G[k] = Gr[k];
          const float normdp = normdp_l1(dp);
          S.dp[6] = normdp;
          S.nv = nv;
          if (trace && trace_n < prm.trace_cap) {
            float* rec = trace + (int64_t)ICT_TRACE_FLOATS * trace_n;
            trace_record(rec, sl, it, sumsd, dp, normdp, nv);
            rec[16] = (float)(tc1 - tc0);          // cycles of the chain loop ...
            rec[17] = (float)tw;                   // ... of which waiting for the producers
            rec[18] = (float)(clock64() - tc1);    // redux, solve, exp
            rec[19] = (float)tcons;                // additions + loads of the chain warp alone
          }
        }
        __syncwarp();
        if (trace && trace_n < prm.trace_cap) ++trace_n;
        const float normdp = S.dp[6];
        nvsum += S.nv;
        if (it == 0) normdp_init = normdp;
        const int cont = keep_iterating(op, it + 1, normdp, normdp_init);
        if (lane == 0) {
          S.it = it + 1;
          S.cont = cont;
        }
      }
      __syncthreads();
      ++it;
    }
    if (chainw && lane == 0) store_level_iters(prm.iters, op, t, sl, S.it);
  }

  if (state) {   // the last iteration ended with a CTA barrier: the arrays are quiescent
    float2* st2 = reinterpret_cast<float2*>(state);
    for (int e = tid; e < 3 * 32 * Q; e += nt) st2[e] = s_ref2[e];
    for (int e = tid; e < 12 * P; e += nt) state[3 * 64 * P + e] = s_AB[e];
  }
  if (chainw && lane == 0) finish_track(prm, t, donorm, S.p, S.G, prm.p_out, prm.npixres, (long long)nvsum * N, trace, trace_n);
}

static int x8_tpp(const ict_optparam& op) { return op.psz == 16 ? 4 : 1; }   // tiles (64 pixels) per patch
static size_t kx8_smem_np(const ict_optparam& op, int max_pts, int np) {
  const size_t P = (size_t)track_pcap(op, max_pts), Q = P * x8_tpp(op);
  return sizeof(float) * (3 * 64 * Q + 2 * np * X8_TILE + 36 * P);
}
static bool x8_form_ok(const ict_optparam& op, int max_pts, int np) {
  return track_pcap(op, max_pts) * x8_tpp(op) <= np * X8_MAXR && kx8_smem_np(op, max_pts, np) <= (size_t)ICT_TRACK_SMEM_LIMIT;
}
size_t kx8_smem_bytes(const ict_optparam& op, int max_pts) {
  return kx8_smem_np(op, max_pts, x8_form_ok(op, max_pts, KX_PROD) ? KX_PROD : 15);
}

// 8x8 patches with or without dopatchnorm; 16x16 patches (four tiles per patch) without
bool kx8_supported(const ict_optparam& op, int max_pts) {
  if (!(op.psz == 8 || (op.psz == 16 && !op.dopatchnorm))) return false;
  return x8_form_ok(op, max_pts, KX_PROD) || x8_form_ok(op, max_pts, 15);
}

template <bool PN, int NP, int TPP, int PK>
static cudaError_t launch_x8_t(const TrackParams& prm, size_t smem, cudaStream_t stream) {
  return launch_cta_kernel<k_track_x8<PN, NP, TPP, PK>>(prm.T, (NP + 1) * 32, smem, 100, stream, prm);
}

template <int PK>
static cudaError_t launch_x8_pk(const TrackParams& prm, bool wide, size_t smem7, size_t smem15, cudaStream_t stream) {
  if (prm.op.psz == 16)
    return wide ? launch_x8_t<false, 15, 4, PK>(prm, smem15, stream) : launch_x8_t<false, 7, 4, PK>(prm, smem7, stream);
  if (wide)
    return prm.op.dopatchnorm ? launch_x8_t<true, 15, 1, PK>(prm, smem15, stream) : launch_x8_t<false, 15, 1, PK>(prm, smem15, stream);
  return prm.op.dopatchnorm ? launch_x8_t<true, 7, 1, PK>(prm, smem7, stream) : launch_x8_t<false, 7, 1, PK>(prm, smem7, stream);
}

cudaError_t launch_track_x8(const TrackParams& prm, int max_pts, cudaStream_t stream) {
  if (prm.T <= 0) return cudaSuccess;
  const size_t smem7 = kx8_smem_np(prm.op, max_pts, 7), smem15 = kx8_smem_np(prm.op, max_pts, 15);
  const bool ok7 = x8_form_ok(prm.op, max_pts, 7), ok15 = x8_form_ok(prm.op, max_pts, 15);
  int sms = 148;
  {
    int dev_ = 0;
    cudaGetDevice(&dev_);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev_);
  }
  // 15 producers where they cost no residency: one CTA per SM anyway (more than 113 KB with 7), or a batch that does not
  // fill the SMs twice
  const bool wide = ok15 && (!ok7 || 2 * (smem7 + 1024) > 228 * 1024 || prm.T <= sms);
  return prm.eigen_packet == 8 ? launch_x8_pk<8>(prm, wide, smem7, smem15, stream)
                               : launch_x8_pk<4>(prm, wide, smem7, smem15, stream);
}

}  // namespace ict
