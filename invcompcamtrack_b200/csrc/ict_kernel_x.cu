// ict_kernel_x.cu — K2x: SetPose + TrackPose for 32x32 patches with the REFERENCE'S ORDER OF SUMMATION
// (ict_tracker_set_sum_order(tr, 1), no patch normalisation): bit-identical to the oracle's default model of the
// reference (Eigen 3.3 vectorised .sum(): 4-float packets, two accumulators — oracle/ictrack_oracle.c
// DEF_PACKET_SUM), like k_track<32, 2> in ict_kernels.cu, but organised so that the sequential chains do not leave
// the rest of the CTA idle.
//
// Eigen's sum of v[0..N) is eight interleaved SEQUENTIAL fp32 chains (chain c adds v[c], v[8+c], v[16+c], ... in
// that order) followed by (c0+c4 + c2+c6) + (c1+c5 + c3+c7).  fp32 addition is not associative, so the chains have
// to be run as written; what CAN be parallel is everything before the additions.  With e = point*1024 + row*32 +
// col, chain c takes the columns c, c+8, c+16, c+24 of every row, points and rows in ascending order.  So:
//
//   * seven PRODUCER warps compute, tile by tile (a tile = four rows of one point, lane = column), the values that
//     get summed — sd_k * pdiff for the six J^T r sums of an iteration, sd_a * sd_b for six of the 21 Hessian sums per
//     pass — with the reference's roundings (sd_k = fl(fl(dx*A_k) + fl(dy*B_k)), unfused bilinear sample, everything
//     compiled with -fmad=false) and store them as float4 row-quads in a staging ring in shared memory;
//   * one CHAIN warp owns the 48 chains of the six sums (lane l: chain (k = l/8, c = l%8) and, for l < 16, chain
//     (k = 4 + l/8, c)); per tile it reads its four columns of the four rows (4 x LDS.128 per chain) and performs
//     the 16 additions in the reference's order;
//   * work proceeds in rounds of seven tiles (producer w makes tile 7j + w of round j) over a two-half staging ring;
//     the halves are handed over with shared-memory barriers (mbarrier: `full[h]` completes when all producers have
//     written their tile of the round, `empty[h]` when the chain warp has read the half), so the producers run one
//     round ahead of the chain warp and nobody waits at a CTA barrier inside a sum; one CTA barrier per iteration
//     remains (the next iteration needs the new pose).  Handing over single tiles instead was slower: every
//     mbarrier wait costs the chain warp ~90 cycles of issue stall, 32 times per sum.
// The chain warp then combines the chains like Eigen's redux, solves with Eigen's elimination (lu6_* of
// ict_device.cuh), updates the pose with the reference's exp (double sqrt/sin/cos, utilities.h:84-145) and places
// the points for the next iteration.  Template layout, gather and placement are those of K2v2 (ict_kernel_v2.cuh),
// which are already reference-exact.
#include "ict_kernels.cuh"
#include "ict_device.cuh"
#include "ict_kernel_v2.cuh"
#include "ict_kernel_x.cuh"

namespace ict {


#define KX_TILE_F4 (6 * 32)             /* float4 per staged tile: six quantities x 32 columns (x 4 rows) */

// One producer tile: rows 4*rq .. 4*rq+3 of point i, this lane's column.  MODE 0..3: Hessian pass (products of
// steepest-descent values); MODE 4: iteration (sd_k * pdiff; pn4 = the four new-frame samples, vis = point visible).
template <int MODE>
__device__ __forceinline__ void kx_produce(const float4 R, const float4 GX, const float4 GY, const float* ab,
                                           const float4 pn4, bool vis, float4* dst /* [6][32] float4, + lane */) {
  const float gx[4] = {GX.x, GX.y, GX.z, GX.w}, gy[4] = {GY.x, GY.y, GY.z, GY.w};
  const float rf[4] = {R.x, R.y, R.z, R.w}, pn[4] = {pn4.x, pn4.y, pn4.z, pn4.w};
  float v[6][4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float sd[6];
    kx_sd(gx[j], gy[j], ab, sd);
    if (MODE == 4) {
      const float pd = vis ? rf[j] - pn[j] : 0.0f;   // pdiff (odometer.cpp:381); 0 where the point is not visible
#pragma unroll
      for (int k = 0; k < 6; ++k) v[k][j] = sd[k] * pd;   // sd_k_proj, odometer.cpp:386-391
    } else {
      float o[6];
      kx_hess_products<MODE>(sd, o);
#pragma unroll
      for (int k = 0; k < 6; ++k) v[k][j] = o[k];
    }
  }
#pragma unroll
  for (int k = 0; k < 6; ++k) dst[k * 32] = make_float4(v[k][0], v[k][1], v[k][2], v[k][3]);
}

// Chain warp, one tile: chain (k, c) adds columns c, c+8, c+16, c+24 of rows 0..3 in that order.  first: this is
// element 0 of the whole sum (Eigen starts a chain with its first packet, it does not add it to zero).
__device__ __forceinline__ void kx_consume(const float4* tile, int lane, bool first, float& sx, float& sy) {
  const int c = lane & 7, kx = lane >> 3;
  const float4* px = tile + kx * 32 + c;
  const float4* py = tile + (4 + kx) * 32 + c;
  const float4 x0 = px[0], x1 = px[8], x2 = px[16], x3 = px[24];
  float4 y0 = make_float4(0.f, 0.f, 0.f, 0.f), y1 = y0, y2 = y0, y3 = y0;
  if (lane < 16) { y0 = py[0]; y1 = py[8]; y2 = py[16]; y3 = py[24]; }
  sx = first ? x0.x : sx + x0.x;  sy = first ? y0.x : sy + y0.x;
  sx = sx + x1.x; sy = sy + y1.x; sx = sx + x2.x; sy = sy + y2.x; sx = sx + x3.x; sy = sy + y3.x;
  sx = sx + x0.y; sy = sy + y0.y; sx = sx + x1.y; sy = sy + y1.y; sx = sx + x2.y; sy = sy + y2.y; sx = sx + x3.y; sy = sy + y3.y;
  sx = sx + x0.z; sy = sy + y0.z; sx = sx + x1.z; sy = sy + y1.z; sx = sx + x2.z; sy = sy + y2.z; sx = sx + x3.z; sy = sy + y3.z;
  sx = sx + x0.w; sy = sy + y0.w; sx = sx + x1.w; sy = sy + y1.w; sx = sx + x2.w; sy = sy + y2.w; sx = sx + x3.w; sy = sy + y3.w;
}

// One round: the tiles 7j .. 7j+6 of a ring half, in order.  A full round is straight-line code (no per-tile test),
// so the loads of the later tiles are issued while the additions of the earlier ones are still in flight.
__device__ __forceinline__ void kx_consume_round(const float4* half, int lane, int j, int ntile, float& sx, float& sy) {
  if ((j + 1) * KX_PROD <= ntile) {
#pragma unroll
    for (int w = 0; w < KX_PROD; ++w) kx_consume(half + w * KX_TILE_F4, lane, w == 0 && j == 0, sx, sy);
  } else {
    for (int w = 0; j * KX_PROD + w < ntile; ++w) kx_consume(half + w * KX_TILE_F4, lane, w == 0 && j == 0, sx, sy);
  }
}

__global__ void __launch_bounds__(256, 2) k_track_x(const TrackParams prm) {
  constexpr int N = 1024;
  extern __shared__ __align__(16) float smem[];
  __shared__ KxShared S;

  const int t = blockIdx.x + prm.t0;
  const ict_optparam& op = prm.op;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
  const int64_t off = prm.pt_off[t];
  const int n_in = (int)(prm.pt_off[t + 1] - off);
  const int P = min(n_in, op.maxpttrack);
  const int E = P * N;
  const int NTILE = 8 * P;
  const bool donorm = op.donorm != 0;

  float4* s_ref4 = reinterpret_cast<float4*>(smem);          // [P][8][32] : rows 4q..4q+3 of column c
  float4* s_gx4 = s_ref4 + E / 4;
  float4* s_gy4 = s_gx4 + E / 4;
  float4* s_ring = s_gy4 + E / 4;                            // [2][KX_PROD] tiles of KX_TILE_F4 float4
  float4* s_rpl = s_ring + 2 * KX_PROD * KX_TILE_F4;         // [P][2] reference placement {base,vis,-,-},{w0..w3}
  float4* s_npl = s_rpl + 2 * P;                             // [KX_PROD][P][2] new-frame placement, one copy per producer
  float* s_AB = reinterpret_cast<float*>(s_npl + 2 * P * KX_PROD);   // [P][12]
  float* s_X = s_AB + 12 * P;
  float* s_Y = s_X + P;
  float* s_Z = s_Y + P;
  float* s_Xc = s_Z + P;
  float* s_Yc = s_Xc + P;
  float* s_Zc = s_Yc + P;

  const TrackFrames fr = track_frames(prm, t);
  const bool chainw = warp == KX_PROD;

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
  if (tid == 0) track_setpose(prm.p_in, prm.norm, t, donorm, S.p, S.G);
  if (tid >= 32 && tid < 34) {
    mbar_init(&S.full[tid - 32], 32 * KX_PROD);
    mbar_init(&S.empty[tid - 32], 32);
  }
  __syncthreads();
  for (int i = tid; i < P; i += nt) save_rotated_point(prm, S.G, off, n_in, i, s_X[i], s_Y[i], s_Z[i], s_Xc, s_Yc, s_Zc);
  __syncthreads();

  float* trace = track_trace(prm, t);
  int trace_n = 0;
  float normdp_init = 1e-10f;
  int nvsum = 0;                  // chain warp only
  int ground = 0;                 // rounds done so far, counted alike by every warp: half = ground & 1, use = ground >> 1
  const int ROUNDS = (NTILE + KX_PROD - 1) / KX_PROD;

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
        pl = patch_place(mx, my, 16, width);
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
    // ---- 4b. template gather (all eight warps, 16 rows of one point each; util_getPatch_grad) ----------------------
    for (int g = warp; g < 2 * P; g += nw) {
      const int i = g >> 1, gp = g & 1;
      const float4 pa = s_rpl[2 * i], pw = s_rpl[2 * i + 1];
      if (__float_as_int(pa.y)) {
        const int tq = (i * 8 + gp * 4) * 32 + lane;
        const int o0 = __float_as_int(pa.x) + (gp * 16 - 1) * width + lane;
        gather_plane<16>(Iref + o0, width, pw, s_ref4 + tq);
        gather_plane<16>(Dxr + o0, width, pw, s_gx4 + tq);
        gather_plane<16>(Dyr + o0, width, pw, s_gy4 + tq);
      }
    }
    __syncthreads();

    // ---- 6. Hessian: 21 reference-order sums in four passes of six (odometer.cpp:428-472) --------------------------
#pragma unroll 1
    for (int pass = 0; pass < 4; ++pass) {
      if (!chainw) {
        for (int j = 0; j < ROUNDS; ++j) {
          const int h = ground & 1, use = ground >> 1;
          if (use > 0) mbar_wait_relaxed(&S.empty[h], (use - 1) & 1);   // the chain warp has read this half's previous round
          const int tl = j * KX_PROD + warp;
          if (tl < NTILE) {
            const int i = tl >> 3;
            const float4 GX = s_gx4[tl * 32 + lane], GY = s_gy4[tl * 32 + lane];
            float ab[12];
#pragma unroll
            for (int k = 0; k < 12; ++k) ab[k] = s_AB[i * 12 + k];
            float4* dst = s_ring + (h * KX_PROD + warp) * KX_TILE_F4 + lane;
            const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
            switch (pass) {
              case 0: kx_produce<0>(z4, GX, GY, ab, z4, true, dst); break;
              case 1: kx_produce<1>(z4, GX, GY, ab, z4, true, dst); break;
              case 2: kx_produce<2>(z4, GX, GY, ab, z4, true, dst); break;
              default: kx_produce<3>(z4, GX, GY, ab, z4, true, dst); break;
            }
          }
          mbar_arrive(&S.full[h]);
          ++ground;
        }
      } else {
        float sx = 0.0f, sy = 0.0f;
        for (int j = 0; j < ROUNDS; ++j) {
          const int h = ground & 1;
          mbar_wait(&S.full[h], (ground >> 1) & 1);
          kx_consume_round(s_ring + h * KX_PROD * KX_TILE_F4, lane, j, NTILE, sx, sy);
          mbar_arrive(&S.empty[h]);
          ++ground;
        }
        const float rx = kx_finish(sx), ry = kx_finish(sy);
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
      float sx = 0.0f, sy = 0.0f;
      long long t_c0 = 0, t_c1 = 0;       // instrumentation (trace records [22], [23]): chain loop, serial section
      if (!chainw) {
        // 7. project_pt + new-frame placement (pose.cpp:307-397, utilities.cpp:65-94), lanes = points.  Every
        // producer computes it for itself into its own copy: the chain warp — the critical resource — is spared the
        // ~130 instructions and the producers have the slack.
        float4* npl = s_npl + warp * 2 * P;
        {
          int nvw = 0;
          for (int i0 = 0; i0 < P; i0 += 32) {
            const int i = i0 + lane;
            int v = 0;
            if (i < P) v = place_point(S.G, s_X[i], s_Y[i], s_Z[i], fx, fy, cx, cy, swo, sho, width, npl + 2 * i);
            nvw += __popc(__ballot_sync(0xffffffffu, v));
          }
          if (warp == 0 && lane == 0) S.nv = nvw;
        }
        __syncwarp();
        // producer state: the new-frame rows of the NEXT tile, fetched one tile ahead so that the L2 round trip is
        // covered by the current tile's arithmetic
        float la[5], lb[5];
        float4 lw = make_float4(0.f, 0.f, 0.f, 0.f);
        bool lvis = false;
#pragma unroll
        for (int r = 0; r < 5; ++r) la[r] = lb[r] = 0.0f;
        auto fetch = [&](int tl) {
          const int i = tl >> 3, rq = tl & 7;
          const float4 pa = npl[2 * i];
          lw = npl[2 * i + 1];
          lvis = __float_as_int(pa.y) != 0;
          if (lvis) {
            const float* pI = Inew + (__float_as_int(pa.x) + (rq * 4 - 1) * width + lane);
#pragma unroll
            for (int r = 0; r < 5; ++r) { la[r] = __ldg(pI + r * width); lb[r] = __ldg(pI + r * width - 1); }
          }
        };
        if (warp < NTILE) fetch(warp);
        for (int j = 0; j < ROUNDS; ++j) {
          const int tl = j * KX_PROD + warp;
          const int h = ground & 1, use = ground >> 1;
          const bool have = tl < NTILE;
          float4 pn4 = make_float4(0.f, 0.f, 0.f, 0.f), R = pn4, GX = pn4, GY = pn4;
          float ab[12];
          bool vis = false;
          if (have) {
            const int i = tl >> 3;
            vis = lvis;
            if (vis) {                   // util_getPatch (utilities.cpp:55-113), unfused, reference order
              pn4.x = ((lw.x * la[1] + lw.y * lb[1]) + lw.z * la[0]) + lw.w * lb[0];
              pn4.y = ((lw.x * la[2] + lw.y * lb[2]) + lw.z * la[1]) + lw.w * lb[1];
              pn4.z = ((lw.x * la[3] + lw.y * lb[3]) + lw.z * la[2]) + lw.w * lb[2];
              pn4.w = ((lw.x * la[4] + lw.y * lb[4]) + lw.z * la[3]) + lw.w * lb[3];
            }
            if (tl + KX_PROD < NTILE) fetch(tl + KX_PROD);
            R = s_ref4[tl * 32 + lane]; GX = s_gx4[tl * 32 + lane]; GY = s_gy4[tl * 32 + lane];
#pragma unroll
            for (int k = 0; k < 12; ++k) ab[k] = s_AB[i * 12 + k];
          }
          // every producer keeps step with the ring, with or without a tile in this round (the arrival counts are per round)
          if (use > 0) mbar_wait_relaxed(&S.empty[h], (use - 1) & 1);
          if (have) kx_produce<4>(R, GX, GY, ab, pn4, vis, s_ring + (h * KX_PROD + warp) * KX_TILE_F4 + lane);
          mbar_arrive(&S.full[h]);
          ++ground;
        }
      } else {
        t_c0 = trace ? clock64() : 0;
        for (int j = 0; j < ROUNDS; ++j) {
          const int h = ground & 1;
          mbar_wait(&S.full[h], (ground >> 1) & 1);
          kx_consume_round(s_ring + h * KX_PROD * KX_TILE_F4, lane, j, NTILE, sx, sy);
          mbar_arrive(&S.empty[h]);
          ++ground;
        }
        t_c1 = trace ? clock64() : 0;
      }

      if (chainw) {
        // 9a. sumsd[k]: Eigen's redux of the eight chains
        const float rx = kx_finish(sx), ry = kx_finish(sy);
        // S.nv reaches this warp through the ring's barriers; an empty track has no rounds, and no visible point
        const int nv = NTILE > 0 ? S.nv : 0;
        if ((lane & 7) == 0) {
          S.sum[lane >> 3] = rx;
          if (lane < 16) S.sum[4 + (lane >> 3)] = ry;
        }
        __syncwarp();
        if (lane == 0) {
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
          if (trace && trace_n < prm.trace_cap) {
            float* rec = trace + (int64_t)ICT_TRACE_FLOATS * trace_n;
            trace_record(rec, sl, it, sumsd, dp, normdp, nv);
            rec[22] = (float)(clock64() - t_c1);   // cycles of the serial section (finish, solve, exp)
            rec[23] = (float)(t_c1 - t_c0);        // cycles the chain warp spent consuming the rounds of this sum
          }
        }
        __syncwarp();
        if (trace && trace_n < prm.trace_cap) ++trace_n;
        const float normdp = S.dp[6];
        if (it == 0) normdp_init = normdp;
        const int cont = keep_iterating(op, it + 1, normdp, normdp_init);
        nvsum += nv;
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

  if (chainw && lane == 0) finish_track(prm, t, donorm, S.p, S.G, prm.p_out, prm.npixres, (long long)nvsum * N, trace, trace_n);
}

size_t kx_smem_bytes(const ict_optparam& op, int max_pts) {
  const size_t P = (size_t)track_pcap(op, max_pts);
  return sizeof(float) * (3 * P * 1024 + 2 * KX_PROD * KX_TILE_F4 * 4 + (32 + 8 * KX_PROD) * P);
}

cudaError_t launch_track_x(const TrackParams& prm, int max_pts, cudaStream_t stream) {
  if (prm.T <= 0) return cudaSuccess;
  const size_t smem = kx_smem_bytes(prm.op, max_pts);
  return launch_cta_kernel<k_track_x>(prm.T, 256, smem, 100, stream, prm);
}

}  // namespace ict
