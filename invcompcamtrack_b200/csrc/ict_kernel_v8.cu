// ict_kernel_v8.cu — K2v8: SetPose + TrackPose for 8x8 patches (the reference's own configuration: psz 8, ~100
// points per track, optionally dopatchnorm — run_io_reprojection_test.cpp:15, run_odometer_test.m:232), default
// (tree) summation order, up to 240 points per track (8 warps up to 128 points, 16 beyond; shared memory bounds
// it), optionally a whole chain of frame steps per launch.  The scheme of K2v2 (ict_kernel_v2.cu) with the roles
// re-cut for many small patches:
//
//  * a warp owns the points w, w+NW, w+2NW, ... of the track (w = warp, NW = 8 or 16 warps) and processes one 8x8 patch per step: lane l
//    takes the pixels (2j, c) and (2j+1, c), j = l/8, c = l%8, so the three rows it needs are loaded once (six
//    read-only loads per plane) and the template of its two pixels is one float2 per plane (3 x LDS.64);
//  * the placement (project_pt + util_getPatch's ceil/floor/weights, unfused, bit-exact pixel indexing) of all the
//    warp's points is computed with lanes = points in ONE pass per iteration (k_track_fast re-derived it per point with
//    all lanes doing the same arithmetic: ~95 instructions x 13 points per warp and iteration);
//  * per-lane sums of dx*r and dy*r are kept PER POINT in registers (the patch loop is unrolled over the warp's 16
//    point slots; two CTAs per SM leave 128 registers per thread), reduced once per iteration by a halving butterfly
//    (32 shuffles for 32 values), folded with the point's coefficients by lanes = points, and reduced to six values
//    per warp; the serial warp adds the eight partials, applies the per-level solve matrix (Gauss-Jordan sweeps,
//    ict_kernel_v2.cuh), updates the pose and evaluates exp and the stop rule;
//  * dopatchnorm (utilities.cpp:111-112, 187-188: the mean of the INTENSITY patch is subtracted, reference and new
//    patch alike) costs one extra warp reduction per patch: a patch never leaves its warp.
//
// Arithmetic class = K2v2's: template gather and everything that decides a pixel index unfused in the reference's
// order; fused multiply-adds only in the new-frame sample and the accumulations.  Bit-exact parity is the general
// kernel k_track<8, 2|3> (sum_order 1).
#include "ict_kernels.cuh"
#include "ict_device.cuh"
#include "ict_kernel_v2.cuh"
#include "ict_kernel_v8.cuh"


namespace ict {


#define V8_MP 16                        /* point slots per warp: 8 warps x 16 = 128, 16 warps x 16 = 256 points */

// 16 per-lane values -> their 16 warp totals, total q in lanes 2q and 2q+1 (halving butterfly: 15 + 1 shuffles)
__device__ __forceinline__ float v8_reduce16(const float* v) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  float a[8], b[4], c[2], d;
  {
    const bool up = (lane & 16) != 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float send = up ? v[j] : v[j + 8], keep = up ? v[j + 8] : v[j];
      a[j] = keep + __shfl_xor_sync(FULL, send, 16);
    }
  }
  {
    const bool up = (lane & 8) != 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float send = up ? a[j] : a[j + 4], keep = up ? a[j + 4] : a[j];
      b[j] = keep + __shfl_xor_sync(FULL, send, 8);
    }
  }
  {
    const bool up = (lane & 4) != 0;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const float send = up ? b[j] : b[j + 2], keep = up ? b[j + 2] : b[j];
      c[j] = keep + __shfl_xor_sync(FULL, send, 4);
    }
  }
  {
    const bool up = (lane & 2) != 0;
    const float send = up ? c[0] : c[1], keep = up ? c[1] : c[0];
    d = keep + __shfl_xor_sync(FULL, send, 2);
  }
  return d + __shfl_xor_sync(FULL, d, 1);
}
// which of the 16 values a lane holds after v8_reduce16: bits (16, 8, 4, 2) of the lane select halves in turn
__device__ __forceinline__ int v8_slot_of_lane(int lane) {
  return ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
}

// NW = warps per track: 8 (up to 128 points, two CTAs per SM) or 16 (up to 256 points, one CTA per SM)
template <bool PN, bool TRACE, int NW>
__global__ void __launch_bounds__(32 * NW, NW == 8 ? 2 : 1) k_track_v8(const TrackParams prm) {
  constexpr int N = 64;
  extern __shared__ __align__(16) float smem[];
  __shared__ V2Shared S;
  __shared__ float s_hpart[NW * 24];
  __shared__ float s_part[2][NW * 8];      // per warp: six J^T r partials + visible points, double-buffered

  const int t = blockIdx.x + prm.t0;
  const ict_optparam& op = prm.op;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int64_t off = prm.pt_off[t];
  const int n_in = (int)(prm.pt_off[t + 1] - off);
  const int P = min(n_in, op.maxpttrack);
  const bool donorm = op.donorm != 0;
  const int j2 = lane >> 3, cc = lane & 7;             // this lane's rows 2*j2, 2*j2+1 and column
  const int mslot = v8_slot_of_lane(lane);              // the point slot whose sums this lane holds after a reduction
  const int ipt = warp + NW * mslot;                    // ... and that point
  const bool fold_lane = (lane & 1) == 0 && ipt < P;    // totals are duplicated in lanes 2q, 2q+1

  float2* s_ref2 = reinterpret_cast<float2*>(smem);    // [P][32]: (row 2j, row 2j+1) of column c, lane = 8j + c
  float2* s_gx2 = s_ref2 + 32 * P;
  float2* s_gy2 = s_gx2 + 32 * P;
  float4* s_rpl = reinterpret_cast<float4*>(s_gy2 + 32 * P);   // [P][2] reference placement
  float4* s_npl = s_rpl + 2 * P;                        // [P][2] new-frame placement
  float4* s_hsum = s_npl + 2 * P;                       // [P] {sum dx*dx, sum dx*dy, sum dy*dy, -}
  float* s_AB = reinterpret_cast<float*>(s_hsum + P);   // [P][12]
  float* s_X = s_AB + 12 * P;
  float* s_Y = s_X + P;
  float* s_Z = s_Y + P;
  float* s_Xc = s_Z + P;
  float* s_Yc = s_Xc + P;
  float* s_Zc = s_Yc + P;

  // A chain of frame steps (ict_track_sequence) runs in ONE launch: a track's step k+1 depends on its own step k only,
  // so the CTA loops over the frames and no step waits for the slowest track of the previous one.  Every step starts
  // from the top (reset, points, SetPose) exactly like a launch of its own: same results bit for bit.
  const int nseq = prm.seq_n > 1 ? prm.seq_n : 1;
  const int nlev = op.lv_f - op.lv_l + 1;
  for (int sq = 0; sq < nseq; ++sq) {
  const TrackFrames fr = track_frames(prm, t, sq * prm.seq_step);
  const double* step_p_in = prm.p_in + (int64_t)sq * 6 * prm.T;
  double* step_p_out = prm.p_out + (int64_t)sq * 6 * prm.T;
  int* step_iters = prm.iters ? prm.iters + (int64_t)sq * prm.T * nlev : nullptr;
  long long* step_npix = prm.npixres ? prm.npixres + (int64_t)sq * prm.T : nullptr;
  const int swarp = 0;

  // ---- ResetOdometer (odometer.cpp:580-609) + points -----------------------------------------------------------------
  {
    const float2 z2 = make_float2(0.f, 0.f);
    for (int e = tid; e < 3 * 32 * P; e += nt) s_ref2[e] = z2;
    const float* q = prm.pt3d + 3 * off;
    for (int i = tid; i < P; i += nt) {
      s_X[i] = q[i];
      s_Y[i] = q[n_in + i];
      s_Z[i] = q[2 * (int64_t)n_in + i];
#pragma unroll
      for (int k = 0; k < 12; ++k) s_AB[i * 12 + k] = 0.0f;
    }
  }
  if (tid == 0) track_setpose(step_p_in, prm.norm, t, donorm, S.p, S.G);
  __syncthreads();
  for (int i = tid; i < P; i += nt) save_rotated_point(prm, S.G, off, n_in, i, s_X[i], s_Y[i], s_Z[i], s_Xc, s_Yc, s_Zc);
  __syncthreads();

  float* trace = TRACE ? track_trace(prm, t) : nullptr;
  int trace_n = 0;
  float pk = 0.0f, normdp_init = 1e-10f;   // serial warp: lane (k + 8j) carries pose coefficient k
  int nvsum = 0;
  if (warp == swarp) pk = (lane & 7) < 6 ? S.p[lane & 7] : 0.0f;

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
        pl = patch_place(mx, my, 4, width, (prm.robust & ICT_ROBUST_FLOOR) != 0);
        float c[10];
        sd_coefs(xc, yc, zc, fx, fy, c);
        float* ab = s_AB + i * 12;       // stale coefficients survive when the point is out of view (SURVEY §9.6)
        ab[0] = c[0]; ab[1] = 0.0f; ab[2] = c[2]; ab[3] = c[4]; ab[4] = c[6]; ab[5] = c[8];
        ab[6] = 0.0f; ab[7] = c[1]; ab[8] = c[3]; ab[9] = c[5]; ab[10] = c[7]; ab[11] = c[9];
      }
      s_rpl[2 * i] = make_float4(__int_as_float(pl.base), __int_as_float(vis), 0.0f, 0.0f);
      s_rpl[2 * i + 1] = make_float4(pl.w0, pl.w1, pl.w2, pl.w3);
    }
    __syncthreads();

    // ---- 4b+6a. template gather (unfused, reference order) and per-point sums of dx*dx, dx*dy, dy*dy ---------------
    for (int i = warp; i < P; i += NW) {
      const float4 pa = s_rpl[2 * i], pw = s_rpl[2 * i + 1];
      float2 gx, gy;
      if (__float_as_int(pa.y)) {
        const int o = __float_as_int(pa.x) + (2 * j2 - 1) * width + cc;
        const V8Rows ri = v8_load(Iref, o, width), rx = v8_load(Dxr, o, width), ry = v8_load(Dyr, o, width);
        float2 r = v8_bilin_exact(ri, pw);
        gx = v8_bilin_exact(rx, pw);
        gy = v8_bilin_exact(ry, pw);
        if (PN && op.dopatchnorm) {      // utilities.cpp:187-188: intensity patch minus its mean
          const float m = v8_warp_total(r.x + r.y) / N;
          r.x = r.x - m;
          r.y = r.y - m;
        }
        s_ref2[i * 32 + lane] = r;
        s_gx2[i * 32 + lane] = gx;
        s_gy2[i * 32 + lane] = gy;
      } else {                           // out of the reference image: the previous level's template stays
        gx = s_gx2[i * 32 + lane];
        gy = s_gy2[i * 32 + lane];
      }
      float sxx = fmaf(gx.y, gx.y, gx.x * gx.x), sxy = fmaf(gx.y, gy.y, gx.x * gy.x), syy = fmaf(gy.y, gy.y, gy.x * gy.x);
      sxx = v8_warp_total(sxx);
      sxy = v8_warp_total(sxy);
      syy = v8_warp_total(syy);
      if (lane == 0) s_hsum[i] = make_float4(sxx, sxy, syy, 0.0f);
    }
    __syncwarp();
    {                                    // Hessian contributions of this warp's points: lanes = points, then 21 warp sums
      float h[21];
#pragma unroll
      for (int k = 0; k < 21; ++k) h[k] = 0.0f;
      const int i = warp + NW * lane;
      if (lane < V8_MP && i < P) {
        const float4 sm = s_hsum[i];
        const float* ab = s_AB + i * 12;
        int k = 0;
#pragma unroll
        for (int a = 0; a < 6; ++a)
#pragma unroll
          for (int b = a; b < 6; ++b) {
            const float Aa = ab[a], Ab = ab[b], Ba = ab[6 + a], Bb = ab[6 + b];
            h[k] = (Aa * Ab) * sm.x + (Aa * Bb + Ba * Ab) * sm.y + (Ba * Bb) * sm.z;
            ++k;
          }
      }
      warp_sum_store<21>(h, &s_hpart[warp * 24]);
    }
    __syncthreads();

    // ---- 6b. Hessian, the level's solve matrix ---------------------------------------------------------------------------
    if (warp == swarp) {
      float hq = 0.0f;
      if (lane < 21) {
        hq = s_hpart[lane];
#pragma unroll
        for (int wv = 1; wv < NW; ++wv) hq = hq + s_hpart[wv * 24 + lane];
      }
      S.Hinv[lane] = 0.0f;
      S.Hinv[32 + lane] = 0.0f;
      __syncwarp();
      sweep6_solve_matrix(hq, S.Hinv);
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
      // 7. project_pt + new-frame placement of this warp's points, lanes = points
      int nv_w = 0;
      {
        float Gr[12];
#pragma unroll
        for (int k = 0; k < 12; ++k) Gr[k] = S.G[k];
        const int i = warp + NW * lane;
        int v = 0;
        if (lane < V8_MP && i < P)
          v = place_point(Gr, s_X[i], s_Y[i], s_Z[i], fx, fy, cx, cy, swo, sho, width, s_npl + 2 * i, 4,
                          (prm.robust & ICT_ROBUST_FLOOR) != 0);
        nv_w = __popc(__ballot_sync(0xffffffffu, v));
      }
      __syncwarp();
      // 8. one patch per step; per-lane sums of dx*pdiff, dy*pdiff per point slot
      float ax[V8_MP], ay[V8_MP];
#pragma unroll
      for (int m = 0; m < V8_MP; ++m) {
        ax[m] = 0.0f;
        ay[m] = 0.0f;
        const int i = warp + NW * m;
        if (i < P) {                                  // uniform across the warp
          const float4 pa = s_npl[2 * i];
          if (__float_as_int(pa.y)) {
            const float4 pw = s_npl[2 * i + 1];
            const V8Rows rn = v8_load(Inew, __float_as_int(pa.x) + (2 * j2 - 1) * width + cc, width);
            const float2 R = s_ref2[i * 32 + lane], GX = s_gx2[i * 32 + lane], GY = s_gy2[i * 32 + lane];
            float2 pn = v8_bilin_fma(rn, pw);
            if (PN && op.dopatchnorm) {               // utilities.cpp:111-112
              const float mn = v8_warp_total(pn.x + pn.y) / N;
              pn.x = pn.x - mn;
              pn.y = pn.y - mn;
            }
            const float p0 = R.x - pn.x, p1 = R.y - pn.y;   // pdiff, odometer.cpp:381
            ax[m] = fmaf(GX.y, p1, GX.x * p0);
            ay[m] = fmaf(GY.y, p1, GY.x * p0);
          }
        }
      }
      // 9a. per point totals (lanes 2q, 2q+1 hold slot mslot), folded with the point's coefficients, six warp sums
      {
        const float axp = v8_reduce16(ax), ayp = v8_reduce16(ay);
        float b6[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) b6[k] = 0.0f;
        if (fold_lane) {
          const float* ab = s_AB + ipt * 12;
#pragma unroll
          for (int k = 0; k < 6; ++k) b6[k] = fmaf(ayp, ab[6 + k], axp * ab[k]);
        }
        float* part = &s_part[it & 1][warp * 8];
        warp_sum6_store(b6, part);
        if (lane == 0) { part[6] = (float)nv_w; part[7] = 0.0f; }
      }
      __syncthreads();

      if (warp == swarp) {
        const unsigned FULL = 0xffffffffu;
        const int k = lane & 7;
        const float4 h0 = *reinterpret_cast<const float4*>(S.Hinv + 8 * k);
        const float2 h1 = *reinterpret_cast<const float2*>(S.Hinv + 8 * k + 4);
        const float* pp = &s_part[it & 1][0];
        float bk = pp[k];                               // fixed order over the eight warps (k = 6: visible points)
#pragma unroll
        for (int wv = 1; wv < NW; ++wv) bk = bk + pp[wv * 8 + k];
        const float b0 = __shfl_sync(FULL, bk, 0), b1 = __shfl_sync(FULL, bk, 1), b2 = __shfl_sync(FULL, bk, 2);
        const float b3 = __shfl_sync(FULL, bk, 3), b4 = __shfl_sync(FULL, bk, 4), b5 = __shfl_sync(FULL, bk, 5);
        const int nv = (int)__shfl_sync(FULL, bk, 6);
        // 9b. delta_p = M * J^T r (Eigen's solve tabulated once per level), 10. p += delta_p, G = exp(p)
        float dpk = fmaf(h1.y, b5, fmaf(h1.x, b4, fmaf(h0.w, b3, fmaf(h0.z, b2, fmaf(h0.y, b1, h0.x * b0)))));
        // opt-in robustness modes (ictrack.h, ict_tracker_set_robust; not parity):
        //   FULL_STEP — the reference's gradients are I(x+1) - I(x-1), twice the derivative (utilities.cpp:30-31), which
        //   makes H four times and J^T r twice too large: every update is HALF a Gauss-Newton step.  Halving the
        //   gradients is exactly doubling delta_p.
        if (prm.robust & ICT_ROBUST_FULL_STEP) dpk = 2.0f * dpk;
        pk = pk + dpk;
        const float* tf = nullptr;     // teacher forcing (tests): continue from the oracle's pose, not from this one
        if (TRACE) {
          if (prm.teacher && trace && trace_n < prm.trace_cap) {
            tf = prm.teacher + ((int64_t)t * prm.trace_cap + trace_n) * 8;
            pk = (lane & 7) < 6 ? tf[lane & 7] : 0.0f;
          }
        }
        const float q0 = __shfl_sync(FULL, pk, 0), q1 = __shfl_sync(FULL, pk, 1), q2 = __shfl_sync(FULL, pk, 2);
        const float q3 = __shfl_sync(FULL, pk, 3), q4 = __shfl_sync(FULL, pk, 4), q5 = __shfl_sync(FULL, pk, 5);
        float normdp = fabsf(dpk);                      // lpNorm<1> in the reference's association order
        normdp = normdp + __shfl_xor_sync(FULL, normdp, 2);
        normdp = normdp + __shfl_xor_sync(FULL, normdp, 1);
        normdp = normdp + __shfl_xor_sync(FULL, normdp, 4);
        if (lane < 6) S.p[lane] = pk;
        float Gr[12];
        Gr[3] = Gr[7] = Gr[11] = 0.0f;
        if (prm.robust & ICT_ROBUST_COMPOSE) {
          //   COMPOSE — the steepest-descent images are derivatives with respect to a twist applied to the CAMERA-FRAME
          //   points (d Xc / d xi = [I | -[Xc]x], odometer.cpp:306-326), i.e. to G <- exp(delta_p) * G; the reference
          //   instead adds delta_p to the coefficients of G (pose.cpp:116-129), which agrees to first order only.
          const float d0 = __shfl_sync(FULL, dpk, 0), d1 = __shfl_sync(FULL, dpk, 1), d2 = __shfl_sync(FULL, dpk, 2);
          const float d3 = __shfl_sync(FULL, dpk, 3), d4 = __shfl_sync(FULL, dpk, 4), d5 = __shfl_sync(FULL, dpk, 5);
          float Go[12], Ex[12];
#pragma unroll
          for (int j = 0; j < 12; ++j) Go[j] = S.G[j];
          if (lane < 6) S.dps[lane] = dpk;
          Ex[3] = Ex[7] = Ex[11] = 0.0f;
          se3_exp_regs(Ex, d0, d1, d2, d3, d4, d5, S.Ex, S.dps);
#pragma unroll
          for (int r = 0; r < 3; ++r) {
#pragma unroll
            for (int c2 = 0; c2 < 3; ++c2) Gr[4 * r + c2] = Ex[4 * r] * Go[c2] + Ex[4 * r + 1] * Go[4 + c2] + Ex[4 * r + 2] * Go[8 + c2];
            Gr[4 * r + 3] = Ex[4 * r] * Go[3] + Ex[4 * r + 1] * Go[7] + Ex[4 * r + 2] * Go[11] + Ex[4 * r + 3];
          }
          __syncwarp();
          if (lane == 0) {                   // the coefficients of the composed pose, for the output and the trace
            double Gd[12], pl6[6];           // in double: the float log (acos of the trace) loses half its digits near identity
#pragma unroll
            for (int j = 0; j < 12; ++j) Gd[j] = (double)Gr[j];
            se3_log<double>(pl6, Gd);
#pragma unroll
            for (int j = 0; j < 6; ++j) S.p[j] = (float)pl6[j];
          }
          __syncwarp();
          pk = (lane & 7) < 6 ? S.p[lane & 7] : 0.0f;
        } else {
          se3_exp_regs(Gr, q0, q1, q2, q3, q4, q5, S.G, S.p);
        }
        if (it == 0) normdp_init = normdp;
        int cont = keep_iterating(op, it + 1, normdp, normdp_init);
        if (TRACE) {
          if (tf) cont = tf[6] != 0.0f;
        }
        if (lane == 0) {
          *reinterpret_cast<float4*>(S.G) = make_float4(Gr[0], Gr[1], Gr[2], Gr[3]);
          *reinterpret_cast<float4*>(S.G + 4) = make_float4(Gr[4], Gr[5], Gr[6], Gr[7]);
          *reinterpret_cast<float4*>(S.G + 8) = make_float4(Gr[8], Gr[9], Gr[10], Gr[11]);
          S.it = it + 1;
          S.cont = cont;
        }
        if (TRACE) {
          if (trace && trace_n < prm.trace_cap) {
            float* rec = trace + (int64_t)ICT_TRACE_FLOATS * trace_n;
            if (lane < 6) { rec[2 + lane] = bk; rec[8 + lane] = dpk; }
            if (lane == 0) {
              rec[0] = (float)sl;
              rec[1] = (float)it;
              rec[14] = normdp;
              rec[15] = (float)nv;
              for (int q = 16; q < ICT_TRACE_FLOATS; ++q) rec[q] = 0.0f;
            }
            ++trace_n;
          }
        }
        nvsum += nv;
      }
      __syncthreads();
      ++it;
    }
    if (tid == 0) store_level_iters(step_iters, op, t, sl, S.it);
  }

  if (warp == swarp && lane == 0) finish_track(prm, t, donorm, S.p, S.G, step_p_out, step_npix, (long long)nvsum * N, trace, trace_n);
  __syncthreads();                         // the step's pose is written (by thread 0, which reads it next) and shared
  }                                        // memory is free for the next step
}

size_t v8_smem_bytes(const ict_optparam& op, int max_pts) {
  const size_t P = (size_t)track_pcap(op, max_pts);
  return sizeof(float) * (3 * 64 * P + 40 * P);
}

bool v8_supported(const ict_optparam& op, int max_pts) {
  return op.psz == 8 && track_pcap(op, max_pts) <= 16 * V8_MP && v8_smem_bytes(op, max_pts) <= (size_t)ICT_TRACK_SMEM_LIMIT;
}

template <bool PN, bool TRACE, int NW>
static cudaError_t launch_v8_t(const TrackParams& prm, size_t smem, cudaStream_t stream) {
  return launch_cta_kernel<k_track_v8<PN, TRACE, NW>>(prm.T, 32 * NW, smem, 100, stream, prm);
}

template <int NW>
static cudaError_t launch_v8_nw(const TrackParams& prm, size_t smem, cudaStream_t stream) {
  const bool pn = prm.op.dopatchnorm != 0;
  if (prm.trace) return pn ? launch_v8_t<true, true, NW>(prm, smem, stream) : launch_v8_t<false, true, NW>(prm, smem, stream);
  return pn ? launch_v8_t<true, false, NW>(prm, smem, stream) : launch_v8_t<false, false, NW>(prm, smem, stream);
}

cudaError_t launch_track_v8(const TrackParams& prm, int max_pts, cudaStream_t stream) {
  if (prm.T <= 0) return cudaSuccess;
  const size_t smem = v8_smem_bytes(prm.op, max_pts);
  const int P = track_pcap(prm.op, max_pts);
  // sixteen warps for more than 128 points (one CTA per SM then anyway)
  return P > 8 * V8_MP ? launch_v8_nw<16>(prm, smem, stream) : launch_v8_nw<8>(prm, smem, stream);
}

}  // namespace ict
