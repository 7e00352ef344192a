// ict_kernel_v2.cu — K2v2, the production form of SetPose + TrackPose for 32x32 patches (tree reductions, no patch
// normalisation): one 256-thread CTA per track, all levels and iterations on device, like k_track_fast
// (ict_kernels.cu), rebuilt around what ncu showed of that kernel (profiles/r01_k_track_fast_ncu_summary.txt):
// 60 issued instructions per pixel-residual and a ~3000-cycle single-lane section per iteration behind a barrier.
//
//  * Template layout.  (pat_ref, pat_dx, pat_dy) stay resident in shared memory (12 B per template pixel), but four
//    consecutive ROWS of one column are one float4: a lane (= patch column) reads the template of four pixels with
//    three conflict-free LDS.128 instead of twelve LDS.32.
//  * Pixel loop.  Per pixel-residual: two read-only loads (the row and its left-shifted copy; the row above is
//    carried in registers), the bilinear sample as one multiply and three EXPLICIT fused multiply-adds in the
//    reference's association order w0*a + w1*b + w2*c + w3*d (utilities.cpp:107), the residual, and two fused
//    multiply-adds into sum(dx*r), sum(dy*r) of the point (the factorised steepest-descent sums of k_track_fast,
//    ict_device.cuh fold_jtr).  About 12 instructions.  The file is compiled with -fmad=false like the rest of the
//    library: everything that decides a pixel INDEX (projection, ceil/floor placement, bounds tests) and the
//    template itself keep the reference's unfused roundings; fused operations appear only where written as fmaf().
//  * Per point, not per warp: the new-frame placement (project_pt + util_getPatch's ceil/floor/weights) of every
//    point is computed once per iteration by the lanes of the serial warp right after the pose update, and the
//    pixel warps read it back (two LDS.128) instead of each re-deriving it (two IEEE divisions and ~60 more
//    instructions per warp per iteration).  Warps reduce only (sum dx*r, sum dy*r) — 10 shuffles — and the six
//    J^T r entries are formed from the per-point sums by six lanes.
//  * Serial section.  Six lanes fold the partial sums directly in the row order of the LU factorisation; lane 0
//    runs the straight-line forward/backward substitution on factors every lane prefetched as float4 before the
//    sums arrive, updates the pose (additive, pose.cpp:116-129), evaluates exp (double Horner series,
//    ict_device.cuh) and the stop rule; then lanes i < P project the points for the next iteration.
//
// Reference semantics kept (SURVEY.md §9): min two iterations per level, centre-only inclusive bounds test, stale
// template/coefficients of points that leave the reference image at a finer level, new-frame-invisible points
// dropping out of J^T r but staying in H, additive se(3) update.  Parity class = that of k_track_fast: J^T r on
// identical inputs within ~1e-7 of sum|sd*r|; trajectories within the spread of the reference's own summation
// orders (tests/test_gpu_parity.py).  Bit-exact parity is k_track<PSZ, 2> (sum_mode 1).
#include "ict_kernels.cuh"
#include "ict_device.cuh"
#include "ict_kernel_v2.cuh"

namespace ict {


template <int KT, int MINB, bool TRACE, int NT>
__global__ void __launch_bounds__(NT, MINB) k_track_v2(const TrackParams prm) {
  constexpr int N = 1024;                 // pixels per patch (psz 32)
  constexpr int GPP = 32 / KT;            // groups (KT rows, lane = column) per point
  constexpr int RQ = KT / 4;              // float4 row-quads per group
  extern __shared__ __align__(16) float smem[];
  __shared__ V2Shared S;

  const int t = blockIdx.x + prm.t0;
  const ict_optparam& op = prm.op;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
  const int64_t off = prm.pt_off[t];
  const int n_in = (int)(prm.pt_off[t + 1] - off);
  const int P = min(n_in, op.maxpttrack);
  const int E = P * N;
  const int G_all = P * GPP;
  const bool donorm = op.donorm != 0;

  // ---- shared-memory carve-up: template planes as float4 row-quads, then the per-point block ---------------------
  float4* s_ref4 = reinterpret_cast<float4*>(smem);          // [P][8][32] : rows 4q..4q+3 of column c
  float4* s_gx4 = s_ref4 + E / 4;
  float4* s_gy4 = s_gx4 + E / 4;
  float4* s_rpl = s_gy4 + E / 4;                             // [P][2] reference placement {base,vis,-,-},{w0..w3}
  float4* s_npl = s_rpl + 2 * P;                             // [P][2] new-frame placement of the coming iteration
  float4* s_hpart = s_npl + 2 * P;                           // [G_all] {sum dx*dx, sum dx*dy, sum dy*dy, -}
  float2* s_part = reinterpret_cast<float2*>(s_hpart + G_all);   // [2][G_all] {sum dx*r, sum dy*r}, double-buffered
  float* s_AB = reinterpret_cast<float*>(s_part + 2 * G_all);    // [P][12]: A_0..A_5, B_0..B_5 (sd_k = dx*A_k + dy*B_k)
  float* s_X = s_AB + 12 * P;                                // per point: world X Y Z, reference-camera Xc Yc Zc
  float* s_Y = s_X + P;
  float* s_Z = s_Y + P;
  float* s_Xc = s_Z + P;
  float* s_Yc = s_Xc + P;
  float* s_Zc = s_Yc + P;

  const TrackFrames fr = track_frames(prm, t);

  // ---- ResetOdometer (odometer.cpp:580-609) + points -----------------------------------------------------------------
  {
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int e = tid; e < 3 * E / 4; e += nt) s_ref4[e] = z4;
    const float* q = prm.pt3d + 3 * off;
    for (int i = tid; i < P; i += nt) {
      s_X[i] = q[i];
      s_Y[i] = q[n_in + i];
      s_Z[i] = q[2 * (int64_t)n_in + i];
#pragma unroll
      for (int k = 0; k < 12; ++k) s_AB[i * 12 + k] = 0.0f;
    }
  }
  if (tid == 0) track_setpose_from(prm, prm.p_in, t, donorm, S.p, S.G, S.Hsum);
  __syncthreads();
  for (int i = tid; i < P; i += nt) save_rotated_point(prm, S.Hsum, off, n_in, i, s_X[i], s_Y[i], s_Z[i], s_Xc, s_Yc, s_Zc);
  __syncthreads();

  float* trace = TRACE ? track_trace(prm, t) : nullptr;
  int trace_n = 0;
  // state of the serial warp (warp 0), identical in all its lanes unless noted
  float pk = 0.0f;              // lane (k + 8j) carries pose coefficient k (0 for k = 6, 7)
  float normdp_init = 1e-10f;
  int nv = 0;                   // points visible in the new frame at the placements of the coming iteration
  int nvsum = 0;                // sum of nv over all iterations done: pixel-residuals = nvsum * 1024
  if (warp == 0) pk = (lane & 7) < 6 ? S.p[lane & 7] : 0.0f;

  for (int sl = op.lv_f; sl >= op.lv_l; --sl) {
    const float fx = prm.cam.fx[sl], fy = prm.cam.fy[sl], cx = prm.cam.cx[sl], cy = prm.cam.cy[sl];
    const float swo = prm.cam.swo[sl], sho = prm.cam.sho[sl];
    const int width = prm.cam.width[sl];
    const float* __restrict__ Iref = fr.ref->I[sl];
    const float* __restrict__ Dxr = fr.ref->dx[sl];
    const float* __restrict__ Dyr = fr.ref->dy[sl];
    const float* __restrict__ Inew = fr.nw->I[sl];

    const long long t_g0 = TRACE ? clock64() : 0;
    // ---- 4a. per point: reference placement + steepest-descent coefficients (odometer.cpp:268-279, 306-326) ------
    for (int i = tid; i < P; i += nt) {
      const float xc = s_Xc[i], yc = s_Yc[i], zc = s_Zc[i];
      const float mx = (xc / zc) * fx + cx, my = (yc / zc) * fy + cy;   // pt2d[sl][i]
      const int vis = (mx >= 0) & (my >= 0) & (mx <= swo) & (my <= sho);
      PatchPlace pl = {0, 0.f, 0.f, 0.f, 0.f};
      if (vis) {
        pl = patch_place(mx, my, 16, width);
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

    // ---- 4b+6a. template gather (util_getPatch_grad, utilities.cpp:115-189: unfused, reference order) and the
    //      per-group sums of dx*dx, dx*dy, dy*dy ---------------------------------------------------------------------
    for (int g = warp; g < G_all; g += nw) {
      const int i = g / GPP, gp = g - i * GPP;
      const float4 pa = s_rpl[2 * i], pw = s_rpl[2 * i + 1];
      const int tq = (i * 8 + gp * RQ) * 32 + lane;
      if (__float_as_int(pa.y)) {
        // one plane at a time, all 2 * (KT + 1) loads of the plane issued before the first use: the gather is bound by
        // the L2 round trip, not by arithmetic, so the number of loads in flight per warp is what matters
        const int o0 = __float_as_int(pa.x) + (gp * KT - 1) * width + lane;
        gather_plane<KT>(Iref + o0, width, pw, s_ref4 + tq);
        gather_plane<KT>(Dxr + o0, width, pw, s_gx4 + tq);
        gather_plane<KT>(Dyr + o0, width, pw, s_gy4 + tq);
      }
      // (a point out of the reference image keeps the previous level's template, SURVEY.md §9.6)
      float sxx = 0.0f, sxy = 0.0f, syy = 0.0f;
#pragma unroll
      for (int jq = 0; jq < RQ; ++jq) {  // this lane's own writes: no barrier needed
        const float4 gx = s_gx4[tq + jq * 32], gy = s_gy4[tq + jq * 32];
        sxx = fmaf(gx.x, gx.x, sxx); sxy = fmaf(gx.x, gy.x, sxy); syy = fmaf(gy.x, gy.x, syy);
        sxx = fmaf(gx.y, gx.y, sxx); sxy = fmaf(gx.y, gy.y, sxy); syy = fmaf(gy.y, gy.y, syy);
        sxx = fmaf(gx.z, gx.z, sxx); sxy = fmaf(gx.z, gy.z, sxy); syy = fmaf(gy.z, gy.z, syy);
        sxx = fmaf(gx.w, gx.w, sxx); sxy = fmaf(gx.w, gy.w, sxy); syy = fmaf(gy.w, gy.w, syy);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        sxx = sxx + __shfl_xor_sync(0xffffffffu, sxx, o);
        sxy = sxy + __shfl_xor_sync(0xffffffffu, sxy, o);
        syy = syy + __shfl_xor_sync(0xffffffffu, syy, o);
      }
      if (lane == 0) s_hpart[g] = make_float4(sxx, sxy, syy, 0.0f);
    }
    __syncthreads();

    // ---- 6b. Hessian from the per-point sums, the level's solve matrix, first placement -----------------------------------
    if (warp == 0) {
      const long long t_lv0 = TRACE ? clock64() : 0;
      if (TRACE && lane == 0) S.gather_cycles = (float)(t_lv0 - t_g0);
      if (lane < 21) {
        int a = 0, b = 0;                // lane-th pair (a <= b) in the order of ComputeHessian (odometer.cpp:430-455)
        {
          int k = lane, len = 6;
          while (k >= len) { k -= len; --len; ++a; }
          b = a + k;
        }
        float h = 0.0f;
        for (int i = 0; i < P; ++i) {
          float sxx = 0.0f, sxy = 0.0f, syy = 0.0f;
          for (int q = 0; q < GPP; ++q) {
            const float4 v = s_hpart[i * GPP + q];
            sxx = q ? sxx + v.x : v.x;
            sxy = q ? sxy + v.y : v.y;
            syy = q ? syy + v.z : v.z;
          }
          const float* ab = s_AB + i * 12;
          const float Aa = ab[a], Ab = ab[b], Ba = ab[6 + a], Bb = ab[6 + b];
          h = h + ((Aa * Ab) * sxx + (Aa * Bb + Ba * Ab) * sxy + (Ba * Bb) * syy);
        }
        S.Hsum[lane] = h;
      }
      S.Hinv[lane] = 0.0f;
      S.Hinv[32 + lane] = 0.0f;
      __syncwarp();
      sweep6_solve_matrix(lane < 21 ? S.Hsum[lane] : 0.0f, S.Hinv);
      float Gr[12];
#pragma unroll
      for (int k = 0; k < 12; ++k) Gr[k] = S.G[k];
      nv = 0;
      for (int i0 = 0; i0 < P; i0 += 32) {
        const int i = i0 + lane;
        int v = 0;
        if (i < P) v = place_point(Gr, s_X[i], s_Y[i], s_Z[i], fx, fy, cx, cy, swo, sho, width, s_npl + 2 * i);
        nv += __popc(__ballot_sync(0xffffffffu, v));
      }
      normdp_init = 1e-10f;              // odometer.cpp:341-342: normdp = normdp_init = 1e-10
      if (lane == 0) {
        S.it = 0;
        S.cont = keep_iterating(op, 0, 1e-10f, 1e-10f);
        if (TRACE) S.lvl_cycles = (float)(clock64() - t_lv0);
      }
    }
    __syncthreads();

    // ---- iterations (odometer.cpp:344-419) ----------------------------------------------------------------------------
    int it = 0;
    while (S.cont) {
      const long long t_it0 = TRACE ? clock64() : 0;   // instrumentation only (trace records [22], [23])
      float2* part = s_part + (it & 1) * G_all;
      for (int g = warp; g < G_all; g += nw) {
        const int i = g / GPP, gp = g - i * GPP;
        const float4 pa = s_npl[2 * i], pw = s_npl[2 * i + 1];
        float ax = 0.0f, ay = 0.0f;                   // sums of dx*pdiff, dy*pdiff over this group
        if (__float_as_int(pa.y)) {                   // uniform across the warp
          const int tq = (i * 8 + gp * RQ) * 32 + lane;
          const float* pI = Inew + (__float_as_int(pa.x) + (gp * KT) * width + lane);
          float c_ = __ldg(pI - width), d_ = __ldg(pI - width - 1);
#pragma unroll
          for (int jq = 0; jq < RQ; ++jq) {
            const float a0 = __ldg(pI), b0 = __ldg(pI - 1);
            pI += width;
            const float a1 = __ldg(pI), b1 = __ldg(pI - 1);
            pI += width;
            const float a2 = __ldg(pI), b2 = __ldg(pI - 1);
            pI += width;
            const float a3 = __ldg(pI), b3 = __ldg(pI - 1);
            pI += width;
            const float4 R = s_ref4[tq + jq * 32], GX = s_gx4[tq + jq * 32], GY = s_gy4[tq + jq * 32];
            // util_getPatch (utilities.cpp:107) with fused multiply-adds, then pdiff = ref - new (odometer.cpp:381)
            const float n0 = fmaf(pw.w, d_, fmaf(pw.z, c_, fmaf(pw.y, b0, pw.x * a0)));
            const float n1 = fmaf(pw.w, b0, fmaf(pw.z, a0, fmaf(pw.y, b1, pw.x * a1)));
            const float n2 = fmaf(pw.w, b1, fmaf(pw.z, a1, fmaf(pw.y, b2, pw.x * a2)));
            const float n3 = fmaf(pw.w, b2, fmaf(pw.z, a2, fmaf(pw.y, b3, pw.x * a3)));
            const float p0 = R.x - n0, p1 = R.y - n1, p2 = R.z - n2, p3 = R.w - n3;
            ax = fmaf(GX.x, p0, ax); ay = fmaf(GY.x, p0, ay);
            ax = fmaf(GX.y, p1, ax); ay = fmaf(GY.y, p1, ay);
            ax = fmaf(GX.z, p2, ax); ay = fmaf(GY.z, p2, ay);
            ax = fmaf(GX.w, p3, ax); ay = fmaf(GY.w, p3, ay);
            c_ = a3; d_ = b3;
          }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            ax = ax + __shfl_xor_sync(0xffffffffu, ax, o);
            ay = ay + __shfl_xor_sync(0xffffffffu, ay, o);
          }
        }
        if (lane == 0) part[g] = make_float2(ax, ay);
      }
      const long long t_par = TRACE ? clock64() : 0;
      __syncthreads();

      // ---- serial section: one warp, every lane active, ~250 instructions --------------------------------------------
      if (warp == 0) {
        const long long t_ser0 = TRACE ? clock64() : 0;
        const unsigned FULL = 0xffffffffu;
        const int k = lane & 7, k6 = k < 6 ? k : 0, j4 = lane >> 3;
        // 9a. J^T r from the per-point sums: sum_k = sum_i (A_ki * ax_i + B_ki * ay_i).  Lane (k + 8j) takes the
        //     points i = j, j+4, ...; two butterfly steps add the four point slots in a fixed order.
        const float4 h0 = *reinterpret_cast<const float4*>(S.Hinv + 8 * k);        // row k of H^-1 (issued early)
        const float2 h1 = *reinterpret_cast<const float2*>(S.Hinv + 8 * k + 4);
        float bk = 0.0f;
        if (P <= 4) {                                  // one point per lane slot: no loop
          if (j4 < P) {
            float2 v = part[j4 * GPP];
#pragma unroll
            for (int q = 1; q < GPP; ++q) {
              const float2 u = part[j4 * GPP + q];
              v.x = v.x + u.x;
              v.y = v.y + u.y;
            }
            bk = fmaf(v.y, s_AB[j4 * 12 + 6 + k6], v.x * s_AB[j4 * 12 + k6]);
          }
        } else {
#pragma unroll 1
          for (int i = j4; i < P; i += 4) {
            float2 v = part[i * GPP];
#pragma unroll
            for (int q = 1; q < GPP; ++q) {
              const float2 u = part[i * GPP + q];
              v.x = v.x + u.x;
              v.y = v.y + u.y;
            }
            bk = bk + fmaf(v.y, s_AB[i * 12 + 6 + k6], v.x * s_AB[i * 12 + k6]);
          }
        }
        bk = bk + __shfl_xor_sync(FULL, bk, 8);
        bk = bk + __shfl_xor_sync(FULL, bk, 16);
        // 9b. delta_p = M * J^T r: Eigen's solve (odometer.cpp:407) tabulated once per level, lane k takes row k
        const float b0 = __shfl_sync(FULL, bk, 0), b1 = __shfl_sync(FULL, bk, 1), b2 = __shfl_sync(FULL, bk, 2);
        const float b3 = __shfl_sync(FULL, bk, 3), b4 = __shfl_sync(FULL, bk, 4), b5 = __shfl_sync(FULL, bk, 5);
        const float dpk = fmaf(h1.y, b5, fmaf(h1.x, b4, fmaf(h0.w, b3, fmaf(h0.z, b2, fmaf(h0.y, b1, h0.x * b0)))));
        // 10. addpose_se3 (pose.cpp:116-129): p += delta_p, G = exp(p)
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
        // lpNorm<1> (odometer.cpp:412) in the reference's order ((|d0|+|d2|) + (|d1|+|d3|)) + (|d4|+|d5|)
        float normdp = fabsf(dpk);
        normdp = normdp + __shfl_xor_sync(FULL, normdp, 2);
        normdp = normdp + __shfl_xor_sync(FULL, normdp, 1);
        normdp = normdp + __shfl_xor_sync(FULL, normdp, 4);
        if (lane < 6) S.p[lane] = pk;
        float Gr[12];
        Gr[3] = Gr[7] = Gr[11] = 0.0f;
        se3_exp_regs(Gr, q0, q1, q2, q3, q4, q5, S.G, S.p);
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
              rec[16] = 0.0f;
              rec[20] = 0.0f;
              rec[17] = (float)(t_ser0 - t_par);         // cycles this warp waited at the barrier for the others
              rec[19] = S.gather_cycles;                 // cycles of this level's placement + template gather
              rec[21] = S.lvl_cycles;                    // cycles of this level's Hessian fold + LU + inverse
              rec[22] = (float)(clock64() - t_ser0);     // cycles of the serial section up to here
              rec[23] = (float)(t_par - t_it0);          // cycles the serial warp spent in the pixel section
            }
          }
        }
        nvsum += nv;
        // 7. project_pt with the new pose + new-frame placement for the next iteration (one point per lane)
        if (cont) {
          nv = 0;
          for (int i0 = 0; i0 < P; i0 += 32) {
            const int i = i0 + lane;
            int v = 0;
            if (i < P) v = place_point(Gr, s_X[i], s_Y[i], s_Z[i], fx, fy, cx, cy, swo, sho, width, s_npl + 2 * i);
            nv += __popc(__ballot_sync(FULL, v));
          }
        }
        if (TRACE) {
          if (trace && trace_n < prm.trace_cap) {
            if (lane == 0) trace[(int64_t)ICT_TRACE_FLOATS * trace_n + 18] = (float)(clock64() - t_ser0);
            ++trace_n;
          }
        }
      }
      __syncthreads();
      ++it;
    }
    // (S.it is next written by the serial warp two barriers further down, in the next level's set-up)
    if (tid == 0) store_level_iters(prm.iters, op, t, sl, S.it);
  }

  if (warp == 0 && lane == 0) finish_track(prm, t, donorm, S.p, S.G, prm.p_out, prm.npixres, (long long)nvsum * N, trace, trace_n);
}

size_t v2_smem_bytes(const ict_optparam& op, int max_pts) {
  const size_t P = (size_t)track_pcap(op, max_pts);
  return sizeof(float) * (3 * P * 1024 + 72 * P);
}

template <int KT, int MINB, bool TRACE, int NT = 256>
static cudaError_t launch_v2_t(const TrackParams& prm, size_t smem, cudaStream_t stream) {
  return launch_cta_kernel<k_track_v2<KT, MINB, TRACE, NT>>(prm.T, NT, smem, 100, stream, prm);
}

cudaError_t launch_track_v2(const TrackParams& prm, int max_pts, cudaStream_t stream) {
  if (prm.T <= 0) return cudaSuccess;
  const size_t smem = v2_smem_bytes(prm.op, max_pts);
  // More points per track = more template per CTA = fewer CTAs per SM: keep ~32 warps per SM by giving the track more
  // warps (a warp still owns 16 rows of one point at a time; per-group sums make the result independent of it).
  const int P = track_pcap(prm.op, max_pts);
  if (P > 8)
    return prm.trace ? launch_v2_t<16, 1, true, 1024>(prm, smem, stream) : launch_v2_t<16, 1, false, 1024>(prm, smem, stream);
  if (P > 4)
    return prm.trace ? launch_v2_t<16, 2, true, 512>(prm, smem, stream) : launch_v2_t<16, 2, false, 512>(prm, smem, stream);
  if (prm.trace) return launch_v2_t<16, 4, true>(prm, smem, stream);   // same arithmetic + per-iteration records
  return launch_v2_t<16, 4, false>(prm, smem, stream);
}

}  // namespace ict
