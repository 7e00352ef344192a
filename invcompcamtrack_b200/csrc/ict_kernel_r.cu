// ict_kernel_r.cu — K2r: SetPose + TrackPose for 32x32 patches in the REFERENCE'S ORDER OF SUMMATION (the library
// default, ict_tracker_set_sum_order(tr, 1)): bit-identical to the oracle's model of the reference (Eigen 3.3
// vectorised .sum(): eight interleaved sequential fp32 chains — oracle/ictrack_oracle.c DEF_PACKET_SUM).
//
// What bounds a reference-order kernel is the chain: chain c of a sum adds its 128 * P elements one after the other
// (fp32 addition is not associative), 4 cycles per addition, so one J^T r costs >= 2048 cycles for a four-point
// track whatever else happens.  Everything is arranged so that nothing but that chain is on the critical path:
//
//   * The six steepest-descent images of the track live in shared memory for the whole level, exactly the arrays the
//     reference keeps (sd1..sd6, odometer.cpp:317-326): 24 B per template pixel, 96 KB for four 32x32 patches, two
//     tracks per SM.  A chain lane's work per element is then one multiplication and its addition — the 14 flops
//     per pixel that re-deriving sd_k from (dx, dy) costs (K2x) are paid once per level.  Layout [point][k][row][c][i]
//     with column = c + 8 i: the four consecutive elements of chain c in a row are one LDS.128.
//   * The 48 chains of J^T r (6 sums x 8) are 48 lanes: chain warp A holds k = 0..3 (lane = 8 k + c), chain warp B
//     k = 4, 5.  Per row a chain lane issues two LDS.128 (its sd quad, the row's pdiff quad), four FMUL, four FADD.
//     The 21 x 8 = 168 chains of the Hessian run the same way on six warps in ONE pass (sd_a quad, sd_b quad).
//   * The new-frame window of every half patch (a "unit": 16 rows of one point) is fetched by ONE 2-D TMA box load
//     (cp.async.bulk.tensor.2d, box 40 x 17 floats from the padded level plane, complete_tx on an mbarrier) straight
//     into shared memory: no per-pixel address arithmetic, no L1 traffic.  Four PRODUCER warps (lane = patch column)
//     turn a window into the unit's pdiff rows IN PLACE (row r of the window is dead once row r of the patch is
//     sampled), with util_getPatch's unfused arithmetic (utilities.cpp:55-113) and the template intensities of
//     their rows in REGISTERS (32 per lane); the chain warps read pdiff from the window slot.  Five slots are
//     recycled over the eight units of a four-point track; every hand-off is an mbarrier (TMA landed -> producer,
//     pdiff written -> chain warps, slot consumed -> next TMA), one CTA barrier per iteration.
//   * The reference template (I, dx, dy windows of odometer.cpp:286) arrives the same way: 3 TMA boxes per unit,
//     staged in the point's own (about to be rewritten) sd area.
//   * Chain warp A then runs the serial section: Eigen's redux of the chains, FullPivLU::solve in Eigen's order with
//     true divisions (lu6_solve_exact), additive update + the reference's exp (pose.cpp:116-129), stop rule, the
//     placement of the points for the next iteration (lanes = points) and the issue of the next windows.
//
// Stale state (odometer.cpp:580-609: arrays are cleared only by Set3Dpoints): a point that is outside the reference
// image at some level keeps the steepest-descent values and the template intensities of the previous level — here
// its sd area and its producers' registers are simply not rewritten.
#include <cuda.h>

#include "ict_kernels.cuh"
#include "ict_device.cuh"
#include "ict_kernel_x.cuh"

namespace ict {

void count_launch_external();

// A window needs 33 columns (the column to the left of the patch + 32).  The box start must be a multiple of four
// floats: with 4-byte elements and no interleave the hardware rejects (illegal instruction) an innermost coordinate
// that is not 16-byte aligned (profiles/tools/probe/tma_probe3.cu; x = 36, 40 work, 37, 38 fault), so the box starts
// at the column rounded down and is 40 wide; the 0..3 extra columns on the left are skipped when sampling.
#define KR_WROW 40                      /* floats per window row */
#define KR_WIN_BYTES (17 * KR_WROW * 4) /* one unit's window: 17 rows (row above + 16) */
#define KR_SLOT_BYTES 2816              /* KR_WIN_BYTES rounded up to the 128-byte TMA destination alignment */
#define KR_NSLOT 5

#define KR_MAXU 16                      /* units per track: 2 per point, up to 8 points */
#define KR_SD_BYTES_PER_POINT (6 * 1024 * 4)

__device__ __forceinline__ void tma_load_2d(void* dst, const void* tmap, int x, int y, unsigned long long* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          ict_saddr(dst)),
      "l"(tmap), "r"(x), "r"(y), "r"(ict_saddr(bar))
      : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_only(unsigned long long* b, unsigned bytes) {   // no arrival
  asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(ict_saddr(b)), "r"(bytes) : "memory");
}
// Producer-side wait for a window: a few immediate polls (the first units' windows are on the critical path of the
// iteration), then a short sleep per poll.  A tight try_wait loop of the waiting producers was 20 % of all issued
// instructions (ncu), on the schedulers the chain warps need.
__device__ __forceinline__ void mbar_wait_backoff(unsigned long long* b, unsigned parity) {
  unsigned done = 0;
  for (int tries = 0;; ++tries) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
        "selp.u32 %0, 1, 0, P1;\n"
        "}\n"
        : "=r"(done)
        : "r"(ict_saddr(b)), "r"(parity)
        : "memory");
    if (done) break;
    if (tries >= 4) __nanosleep(40);
  }
}
// generic-proxy accesses to shared memory (the in-place pdiff stores, the chain warps' loads) ordered before the
// async-proxy write of the next TMA into the same slot
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// the tensor maps live in global memory (one per frame, plane and level, written by the host at store creation)
// and were copied there by cudaMemcpy: every thread that issues a TMA with a map acquires it first (system scope)
__device__ __forceinline__ void tmap_acquire(const void* tmap) {
  asm volatile("fence.proxy.tensormap::generic.acquire.sys [%0], 128;" ::"l"(tmap) : "memory");
}

struct __align__(16) KrShared {
  unsigned long long win_full[KR_MAXU];    // unit's window landed (TMA complete_tx) or unit not visible: 1 arrival
  unsigned long long slot_free[KR_MAXU];   // unit's pdiff consumed by its two chain warps: 2 arrivals
  unsigned long long gat_full[2];          // reference windows of a level landed: points 0..3 / points 4..7
  unsigned pd_flag[KR_MAXU];               // serial number of the iteration whose pdiff rows of the unit are written
  unsigned b_flag;                         // ... in which chain warp B has published its two sums
  unsigned pad_[3];
  float G[12];
  float p[8];
  float sum[8];
  float dp[8];
  float Hsum[24];
  Lu6 f;
  float4 npl[8];                           // new-frame bilinear weights per point
  float4 rpl[8];                           // reference-frame weights per point
  int nx[8], ny[8], nvis[8];               // new-frame patch origin (padded plane coordinates), visibility
  int rx[8], ry[8], rvis[8];
  float X[8], Y[8], Z[8], Xc[8], Yc[8], Zc[8];
  int cont[2], it, nv;                     // cont[gi & 1]: written for the next iteration while the current flag is read
};

// util_getPatch / util_getPatch_grad placement (utilities.cpp:65-94, 127-157): patch origin (column x0, row y0 of the
// padded plane) and the four constant weights.  Unfused, the reference's operation order.
__device__ __forceinline__ void kr_patch_place(float mx, float my, int* x0, int* y0, float4* w) {
  const int pos0 = (int)ceilf(mx + .00001f);
  const int pos1 = (int)ceilf(my + .00001f);
  const int pos2 = (int)floorf(mx);
  const int pos3 = (int)floorf(my);
  const float r0 = mx - (float)pos2;
  const float r1 = my - (float)pos3;
  w->x = r0 * r1;
  w->y = (1 - r0) * r1;
  w->z = r0 * (1 - r1);
  w->w = (1 - r0) * (1 - r1);
  *x0 = pos0 + 16;
  *y0 = pos1 + 16;
}

// 16 bilinear samples of one patch column from a unit's window (row j of the window = image row y0 - 1 + j, column
// lane + 1 of the window = the patch column): ((w0*a + w1*b) + w2*c) + w3*d, utilities.cpp:107,181-183
__device__ __forceinline__ void kr_sample16(const float* win, int lane, const float4 w, float* out) {
  float a0 = win[lane + 1], b0 = win[lane];
#pragma unroll
  for (int r = 0; r < 16; ++r) {
    const float a1 = win[(r + 1) * KR_WROW + lane + 1], b1 = win[(r + 1) * KR_WROW + lane];
    out[r] = ((w.x * a1 + w.y * b1) + w.z * a0) + w.w * b0;
    a0 = a1;
    b0 = b1;
  }
}

// Hand-offs that are on the critical path of an iteration are plain shared-memory flags (release store / acquire
// load, ~30 cycles) instead of mbarriers (a try_wait costs ~90 cycles even when the phase is already complete); a
// flag holds the serial number of the iteration it was last set in.
__device__ __forceinline__ unsigned ld_acquire_s(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"(ict_saddr(p)) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_s(unsigned* p, unsigned v) {
  asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(ict_saddr(p)), "r"(v) : "memory");
}

// Eight rows of a chain: the 32 products first (independent), then the 32 additions in the reference's order.  Written
// as two halves of a unit so that the loads and products of the second half sit in the shadow of the first half's
// dependent additions (4 cycles each).
struct KrRows8 {
  float4 v[8];
};
// ptxas keeps only ~3 rows of loads in flight if left to itself, which does not cover the LDS.128 latency when four
// chain warps and the producers share the SM's shared-memory pipe (measured: 35-45 cycles per row instead of 16).  The
// loads are therefore volatile asm statements: they stay in program order, all sixteen of a half unit up front.
__device__ __forceinline__ float4 lds128v(const float4* p) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(ict_saddr(p)));
  return v;
}
struct KrLoad8 {
  float4 a[8], b[8];
};
__device__ __forceinline__ void kr_load8(const float4* a4, int astride, const float4* b4, int bstride, KrLoad8& o) {
#pragma unroll
  for (int r = 0; r < 8; ++r) { o.a[r] = lds128v(a4 + r * astride); o.b[r] = lds128v(b4 + r * bstride); }
}
__device__ __forceinline__ void kr_mul8(const KrLoad8& l, KrRows8& o) {
#pragma unroll
  for (int r = 0; r < 8; ++r)
    o.v[r] = make_float4(l.a[r].x * l.b[r].x, l.a[r].y * l.b[r].y, l.a[r].z * l.b[r].z, l.a[r].w * l.b[r].w);
}
__device__ __forceinline__ void kr_add8(const KrRows8& p, float& acc) {
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    acc = acc + p.v[r].x;
    acc = acc + p.v[r].y;
    acc = acc + p.v[r].z;
    acc = acc + p.v[r].w;
  }
}

template <int NPROD, int UPP>
__global__ void __launch_bounds__((NPROD + 2) * 32, NPROD == 4 ? 2 : 1) k_track_r(const TrackParams prm) {
  extern __shared__ unsigned char smem_raw[];
  const int t = blockIdx.x + prm.t0;
  const ict_optparam& op = prm.op;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int64_t off = prm.pt_off[t];
  const int n_in = (int)(prm.pt_off[t + 1] - off);
  const int P = min(n_in, op.maxpttrack);
  const int U = 2 * P;
  const bool donorm = op.donorm != 0;

  // shared memory: [sd area: P x 24 KB][window slots: 5 x 2816][KrShared], 128-byte aligned for the TMA destinations
  unsigned char* base = smem_raw + ((128u - (ict_saddr(smem_raw) & 127u)) & 127u);
  float* s_sd = reinterpret_cast<float*>(base);
  const int Pcap = prm.r_pcap;
  unsigned char* s_slots = base + (size_t)Pcap * KR_SD_BYTES_PER_POINT;
  KrShared& S = *reinterpret_cast<KrShared*>(s_slots + KR_NSLOT * KR_SLOT_BYTES);
  float(*s_AB)[12] = reinterpret_cast<float(*)[12]>(s_slots);   // per-point sd coefficients: only live during a level's
                                                                 // precompute, when no window slot is in use

  const int rf = prm.ref_frame ? prm.ref_frame[t] : prm.fixed_ref;
  const int nf = prm.new_frame ? prm.new_frame[t] : prm.fixed_new;
  const char* tm_ref = reinterpret_cast<const char*>(prm.frames[rf].tmap);
  const char* tm_new = reinterpret_cast<const char*>(prm.frames[nf].tmap);
  // role 0: chain warp A (sums 0..3, lane = 8 k + c) and the serial section; role 1: chain warp B (sums 4, 5); the rest
  // produce
  const bool chainA = warp == 0, prod = warp >= 2;
  const int pw = warp - 2;

  // ---- ResetOdometer (odometer.cpp:580-609) + points -------------------------------------------------------------
  {
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    float4* sd4 = reinterpret_cast<float4*>(s_sd);
    for (int e = tid; e < P * (KR_SD_BYTES_PER_POINT / 16); e += nt) sd4[e] = z4;
    const float* q = prm.pt3d + 3 * off;
    for (int i = tid; i < P; i += nt) {
      S.X[i] = q[i];
      S.Y[i] = q[n_in + i];
      S.Z[i] = q[2 * (int64_t)n_in + i];
    }
  }
  if (tid == 0)
    setpose_se3(prm.p_in + 6 * (int64_t)t, donorm, prm.norm + 4 * (int64_t)t, prm.norm[4 * (int64_t)t + 3], S.p, S.G);
  if (tid >= 32 && tid < 32 + KR_MAXU) {
    mbar_init(&S.win_full[tid - 32], 1);
    S.pd_flag[tid - 32] = 0u;
    mbar_init(&S.slot_free[tid - 32], 2);

  }
  if (tid == 64) {
    mbar_init(&S.gat_full[0], 1);
    mbar_init(&S.gat_full[1], 1);
    S.b_flag = 0u;

  }
  mbar_fence_init();
  __syncthreads();
  for (int i = tid; i < P; i += nt) {   // project_pt_save_rotated, pose.cpp:400-488
    const float X = S.X[i], Y = S.Y[i], Z = S.Z[i];
    const float xc = S.G[0] * X + S.G[1] * Y + S.G[2] * Z + S.G[3];
    const float yc = S.G[4] * X + S.G[5] * Y + S.G[6] * Z + S.G[7];
    const float zc = S.G[8] * X + S.G[9] * Y + S.G[10] * Z + S.G[11];
    S.Xc[i] = xc;
    S.Yc[i] = yc;
    S.Zc[i] = zc;
    if (prm.pt2d_out) {
      const int l = op.lv_l;
      prm.pt2d_out[2 * off + i] = (xc / zc) * prm.cam.fx[l] + prm.cam.cx[l];
      prm.pt2d_out[2 * off + n_in + i] = (yc / zc) * prm.cam.fy[l] + prm.cam.cy[l];
    }
  }
  __syncthreads();

  float* trace = prm.trace ? prm.trace + (int64_t)t * prm.trace_cap * ICT_TRACE_FLOATS : nullptr;
  int trace_n = 0;
  float normdp_init = 1e-10f;
  int nvsum = 0;                  // chain warp A only
  unsigned gi = 0;                // iterations so far, counted alike by every warp: parity of the per-unit barriers
  unsigned lvl = 0;               // levels so far: parity of gat_full
  float refv[UPP][16];            // producers: template intensities (pat_ref) of their units' rows, this lane's column
#pragma unroll
  for (int s = 0; s < UPP; ++s)
#pragma unroll
    for (int r = 0; r < 16; ++r) refv[s][r] = 0.0f;
  const int perm = 4 * (lane & 7) + (lane >> 3);   // column -> word of a row in [c][i] order, column = c + 8 i

  for (int sl = op.lv_f; sl >= op.lv_l; --sl, ++lvl) {
    const float fx = prm.cam.fx[sl], fy = prm.cam.fy[sl], cx = prm.cam.cx[sl], cy = prm.cam.cy[sl];
    const float swo = prm.cam.swo[sl], sho = prm.cam.sho[sl];
    const void* tmI = tm_ref + 128 * (0 * ICT_MAX_LEVELS + sl);
    const void* tmDx = tm_ref + 128 * (1 * ICT_MAX_LEVELS + sl);
    const void* tmDy = tm_ref + 128 * (2 * ICT_MAX_LEVELS + sl);
    const void* tmN = tm_new + 128 * (0 * ICT_MAX_LEVELS + sl);

    long long lt0 = 0, lt1 = 0, lt2 = 0, lt3 = 0, lt4 = 0;   // instrumentation (chain warp A, trace only): level phases
    if (chainA && trace) lt0 = clock64();
    // every thread that will issue a TMA with one of this level's maps acquires it once
    if (warp == 0) {
      tmap_acquire(tmI);
      tmap_acquire(tmDx);
      tmap_acquire(tmDy);
      tmap_acquire(tmN);
    } else if (prod && lane == 0) {
      tmap_acquire(tmN);
    }

    // new-frame placement of all points with the current pose + issue of the first KR_NSLOT windows (warp A)
    auto place_and_issue = [&]() {
      int v = 0;
      if (lane < P) {
        const float X = S.X[lane], Y = S.Y[lane], Z = S.Z[lane];
        const float tx = S.G[0] * X + S.G[1] * Y + S.G[2] * Z + S.G[3];       // project_pt, pose.cpp:307-397
        const float ty = S.G[4] * X + S.G[5] * Y + S.G[6] * Z + S.G[7];
        const float tz = S.G[8] * X + S.G[9] * Y + S.G[10] * Z + S.G[11];
        const float mx = (tx / tz) * fx + cx, my = (ty / tz) * fy + cy;
        v = (mx >= 0) & (my >= 0) & (mx <= swo) & (my <= sho);                 // odometer.cpp:369-371 (NaN -> outside)
        int x0 = 0, y0 = 0;
        float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
        if (v) kr_patch_place(mx, my, &x0, &y0, &w);
        S.npl[lane] = w;
        S.nx[lane] = x0;
        S.ny[lane] = y0;
        S.nvis[lane] = v;
      }
      const int nv = __popc(__ballot_sync(0xffffffffu, v));
      if (lane == 0) S.nv = nv;
      __syncwarp();
      if (lane < U && lane < KR_NSLOT) {
        const int pp = lane >> 1, half = lane & 1;
        if (S.nvis[pp]) {
          fence_proxy_async();
          mbar_expect_tx(&S.win_full[lane], KR_WIN_BYTES);
          tma_load_2d(s_slots + lane * KR_SLOT_BYTES, tmN, (S.nx[pp] - 1) & ~3, S.ny[pp] - 1 + 16 * half, &S.win_full[lane]);
        } else {
          mbar_arrive(&S.win_full[lane]);
        }
      }
    };

    // ---- 4a. per point: reference placement + steepest-descent coefficients (odometer.cpp:268-279, 306-326) ------
    if (tid < P) {
      const int i = tid;
      const float xc = S.Xc[i], yc = S.Yc[i], zc = S.Zc[i];
      const float mx = (xc / zc) * fx + cx, my = (yc / zc) * fy + cy;
      const int vis = (mx >= 0) & (my >= 0) & (mx <= swo) & (my <= sho);
      int x0 = 0, y0 = 0;
      float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
      if (vis) {
        kr_patch_place(mx, my, &x0, &y0, &w);
        float c[10];
        sd_coefs(xc, yc, zc, fx, fy, c);
        float* ab = s_AB[i];
        ab[0] = c[0]; ab[1] = 0.0f; ab[2] = c[2]; ab[3] = c[4]; ab[4] = c[6]; ab[5] = c[8];
        ab[6] = 0.0f; ab[7] = c[1]; ab[8] = c[3]; ab[9] = c[5]; ab[10] = c[7]; ab[11] = c[9];
      }
      S.rpl[i] = w;
      S.rx[i] = x0;
      S.ry[i] = y0;
      S.rvis[i] = vis;
    }
    fence_proxy_async();   // generic-proxy accesses to the sd areas so far, before the TMA writes into them
    __syncthreads();
    // ---- 4b. reference windows: three TMA boxes per visible unit into the point's own sd area ---------------------
    if (warp == 0) {
      // every issuing lane adds its own 3 boxes to the transaction count of its barrier, lanes 0 and 1 then make the one
      // arrival of each; two barriers, four points each, keep a barrier's pending transaction count below 64 KB
      if (lane < U && S.rvis[lane >> 1]) {
        const int pp = lane >> 1, half = lane & 1;
        unsigned char* dst = reinterpret_cast<unsigned char*>(s_sd) + (size_t)pp * KR_SD_BYTES_PER_POINT + half * 3 * KR_SLOT_BYTES;
        const int x = (S.rx[pp] - 1) & ~3, y = S.ry[pp] - 1 + 16 * half;
        fence_proxy_async();
        unsigned long long* bar = &S.gat_full[pp >> 2];
        mbar_expect_tx_only(bar, 3u * KR_WIN_BYTES);
        tma_load_2d(dst, tmI, x, y, bar);
        tma_load_2d(dst + KR_SLOT_BYTES, tmDx, x, y, bar);
        tma_load_2d(dst + 2 * KR_SLOT_BYTES, tmDy, x, y, bar);
      }
      __syncwarp();
      if (lane < 2) mbar_arrive(&S.gat_full[lane]);
    }
    if (chainA && trace) lt1 = clock64();
    // ---- 4c/5. template gather (util_getPatch_grad, utilities.cpp:115-189) and steepest-descent values ------------
    float gx[UPP][16], gy[UPP][16];
    if (prod) {
      mbar_wait(&S.gat_full[0], lvl & 1);
      mbar_wait(&S.gat_full[1], lvl & 1);
#pragma unroll
      for (int s = 0; s < UPP; ++s) {
        const int u = pw + NPROD * s;
        if (u < U && S.rvis[u >> 1]) {
          const int pp = u >> 1, half = u & 1;
          const float* win = s_sd + (size_t)pp * (KR_SD_BYTES_PER_POINT / 4) + half * 3 * (KR_SLOT_BYTES / 4) +
                             ((S.rx[pp] - 1) & 3);
          const float4 w = S.rpl[pp];
          kr_sample16(win, lane, w, refv[s]);
          kr_sample16(win + KR_SLOT_BYTES / 4, lane, w, gx[s]);
          kr_sample16(win + 2 * (KR_SLOT_BYTES / 4), lane, w, gy[s]);
        }
      }
    }
    __syncthreads();   // every window has been read: the sd areas may be rewritten
    if (prod) {
#pragma unroll
      for (int s = 0; s < UPP; ++s) {
        const int u = pw + NPROD * s;
        if (u < U && S.rvis[u >> 1]) {
          const int pp = u >> 1, half = u & 1;
          float ab[12];
#pragma unroll
          for (int k = 0; k < 12; ++k) ab[k] = s_AB[pp][k];
          float* dst = s_sd + (size_t)pp * 6 * 1024 + half * 16 * 32 + perm;
#pragma unroll
          for (int r = 0; r < 16; ++r) {
            float sd[6];
            kx_sd(gx[s][r], gy[s][r], ab, sd);
#pragma unroll
            for (int k = 0; k < 6; ++k) dst[k * 1024 + r * 32] = sd[k];
          }
        }
      }
    }
    __syncthreads();

    if (chainA && trace) lt2 = clock64();
    // ---- 6. Hessian: 21 reference-order sums, one chain per lane on six warps (odometer.cpp:428-472) ---------------
    // Three warps, three lane groups of eight chains (c = lane & 7) each; a group's sums share its sd planes, so a row
    // costs eight LDS.128 for the 21 sums instead of twelve and no warp issues more than three of them (a warp gets a
    // shared-memory load issued only every 7-10 cycles; an LDS.128 occupies the SM's pipe for four cycles whatever its
    // lanes read), with one formula per warp (no selects, no divergence):
    //   role 0, group g = 0..2, planes x = 2g, y = 2g + 1:                                 (x,x) (x,y) (y,y)
    //   role 1, group g: plane pairs {0,1}x{2,3}, {0,1}x{4,5}, {2,3}x{4,5}, x = first of the left pair:  (x,z) (x,w)
    //   role 2, the same groups, x = second of the left pair:                              (x,z) (x,w)
    // Lanes 24..31 mirror group 2.
    if (warp < 3) {
      const int c = lane & 7, g = min(lane >> 3, 2);
      auto qidx = [](int a, int b) { return a * 6 - (a * (a - 1)) / 2 + (b - a); };   // position in ComputeHessian's order
      const float4* sd4 = reinterpret_cast<const float4*>(s_sd) + c;
      if (warp == 0) {
        const int px = 2 * g, py = 2 * g + 1;
        const float4* X4 = sd4 + px * 256;
        const float4* Y4 = sd4 + py * 256;
        float a1 = -0.0f, a2 = -0.0f, a3 = -0.0f;   // -0 + x == x for every x: a chain starts with its first element
        for (int i = 0; i < P; ++i) {
#pragma unroll 8
          for (int r = 0; r < 32; ++r) {
            const float4 x = X4[i * 1536 + r * 8], y = Y4[i * 1536 + r * 8];
            a1 = a1 + x.x * x.x; a2 = a2 + x.x * y.x; a3 = a3 + y.x * y.x;
            a1 = a1 + x.y * x.y; a2 = a2 + x.y * y.y; a3 = a3 + y.y * y.y;
            a1 = a1 + x.z * x.z; a2 = a2 + x.z * y.z; a3 = a3 + y.z * y.z;
            a1 = a1 + x.w * x.w; a2 = a2 + x.w * y.w; a3 = a3 + y.w * y.w;
          }
        }
        const float r1 = kx_finish(a1), r2 = kx_finish(a2), r3 = kx_finish(a3);
        if ((lane & 7) == 0 && lane < 24) {
          S.Hsum[qidx(px, px)] = r1;
          S.Hsum[qidx(px, py)] = r2;
          S.Hsum[qidx(py, py)] = r3;
        }
      } else {
        const int px = (g < 2 ? 0 : 2) + (warp - 1), pz = g == 0 ? 2 : 4;
        const float4* X4 = sd4 + px * 256;
        const float4* Z4 = sd4 + pz * 256;
        const float4* W4 = Z4 + 256;
        float a1 = -0.0f, a2 = -0.0f;
        for (int i = 0; i < P; ++i) {
#pragma unroll 8
          for (int r = 0; r < 32; ++r) {
            const float4 x = X4[i * 1536 + r * 8], z = Z4[i * 1536 + r * 8], w = W4[i * 1536 + r * 8];
            a1 = a1 + x.x * z.x; a2 = a2 + x.x * w.x;
            a1 = a1 + x.y * z.y; a2 = a2 + x.y * w.y;
            a1 = a1 + x.z * z.z; a2 = a2 + x.z * w.z;
            a1 = a1 + x.w * z.w; a2 = a2 + x.w * w.w;
          }
        }
        const float r1 = kx_finish(a1), r2 = kx_finish(a2);
        if ((lane & 7) == 0 && lane < 24) {
          S.Hsum[qidx(px, pz)] = r1;
          S.Hsum[qidx(px, pz + 1)] = r2;
        }
      }
    }
    fence_proxy_async();   // the sd coefficients in slot 0, before the first window lands there
    __syncthreads();
    // ---- factorisation (Hes.fullPivLu(), odometer.cpp:514; once per level: the matrix does not change) -------------
    if (chainA && trace) lt3 = clock64();
    if (chainA) {
      lu6_factor_warp(S.Hsum, S.f);

      normdp_init = 1e-10f;              // odometer.cpp:341-342
      const int cont0 = (0 < op.maxiter) & ((1e-10f / 1e-10f) > op.normdp_ratio);
      if (lane == 0) {
        S.it = 0;
        S.cont[gi & 1u] = cont0;
      }
      if (cont0) place_and_issue();
      if (trace) lt4 = clock64();
    }
    __syncthreads();

    // ---- iterations (odometer.cpp:344-419) ----------------------------------------------------------------------------
    int it = 0;
    while (S.cont[gi & 1u]) {
      const unsigned par = gi & 1u;
      if (prod) {
        // 8. new-frame patches + residual (util_getPatch utilities.cpp:55-113, odometer.cpp:381), in place in the window
#pragma unroll
        for (int s = 0; s < UPP; ++s) {
          const int u = pw + NPROD * s;
          if (u < U) {
            const int pp = u >> 1, half = u & 1;
            float* win = reinterpret_cast<float*>(s_slots + (u % KR_NSLOT) * KR_SLOT_BYTES);
            const int vis = S.nvis[pp];
            if (u >= KR_NSLOT) {          // the slot is still in use by unit u - KR_NSLOT: fetch when it is released
              if (lane == 0) {
                mbar_wait_relaxed(&S.slot_free[u - KR_NSLOT], par);
                if (vis) {
                  fence_proxy_async();
                  mbar_expect_tx(&S.win_full[u], KR_WIN_BYTES);
                  tma_load_2d(win, tmN, (S.nx[pp] - 1) & ~3, S.ny[pp] - 1 + 16 * half, &S.win_full[u]);
                } else {
                  mbar_arrive(&S.win_full[u]);
                }
              }
              __syncwarp();
            }
            if (vis) {
              const float4 w = S.npl[pp];
              const float* wsh = win + ((S.nx[pp] - 1) & 3);   // the patch's left neighbour column inside the box
              mbar_wait_backoff(&S.win_full[u], par);
              // The residual rows go back INTO the window (row r of the patch over row r of the window, which only the
              // sample of row r reads), at other word positions than the lanes read: every lane first loads all it
              // needs, the warp synchronises, then it stores — lanes of a warp are not guaranteed to run in lockstep
              // (they leave the barrier wait above one by one), and a lane that stored early would be sampled by its
              // neighbours.
              float a[17], b[17];
#pragma unroll
              for (int r = 0; r < 17; ++r) {
                a[r] = wsh[r * KR_WROW + lane + 1];
                b[r] = wsh[r * KR_WROW + lane];
              }
              __syncwarp();
#pragma unroll
              for (int r = 0; r < 16; ++r) {
                const float pn = ((w.x * a[r + 1] + w.y * b[r + 1]) + w.z * a[r]) + w.w * b[r];
                win[r * KR_WROW + perm] = refv[s][r] - pn;      // pdiff, odometer.cpp:381
              }
            } else {
#pragma unroll
              for (int r = 0; r < 16; ++r) win[r * KR_WROW + perm] = 0.0f;   // sd_proj stays zero (odometer.cpp:352-357)
            }
            // No proxy fence here.  The next write to this slot is a TMA (async proxy), but it is issued by a lane that
            // first acquires slot_free[u] — released by the chain warps after they have READ these stores — and then
            // executes fence.proxy.async itself: the stores are ordered before that fence by the release/acquire chain.
            // A fence.proxy.async per producer lane and unit here sat on the path to every unit's flag: 5 % of the kernel.
            __syncwarp();
            if (lane == 0) st_release_s(&S.pd_flag[u], gi + 1u);
          }
        }
      } else {
        // 9a. the 48 chains of J^T r: lane (k, c) adds sd_k * pdiff over its columns c, c+8, c+16, c+24 of every row
        // (chain warp A: k = 0..3; chain warp B: k = 4, 5, its upper half mirrors the lower).  What bounds this loop is not
        // the four dependent additions per row (16 cycles) but the two LDS.128 that feed them: a warp gets a
        // shared-memory load issued only every 7-10 cycles (profiles/tools/probe/lds_probe2.cu), which with the loads'
        // latency comes to 35-45 cycles per row.  One warp for all 48 chains (three loads per row) and four warps taking
        // turns unit by unit were both measured slower than this split.
        const int c = lane & 7;
        const int k = chainA ? (lane >> 3) : 4 + ((lane >> 3) & 1);
        const float4* sdk = reinterpret_cast<const float4*>(s_sd) + k * 256 + c;
        float acc = -0.0f;   // -0 + x == x for every x: the chain starts with its first element (Eigen's redux)
        long long t_c0 = 0, t_c1 = 0, w0 = 0;   // instrumentation (chain warp A, trace only)
        const unsigned want = gi + 1u;
        if (chainA && trace) t_c0 = clock64();
        if (U > 0)   // an empty track has no unit whose producer would ever raise the flag
          while (ld_acquire_s(&S.pd_flag[0]) != want) {}
        if (chainA && trace) w0 = clock64() - t_c0;
#pragma unroll 1
        for (int u = 0; u < U; ++u) {
          const float4* pd4 = reinterpret_cast<const float4*>(s_slots + (u % KR_NSLOT) * KR_SLOT_BYTES) + c;
          const float4* sd4 = sdk + (u >> 1) * 1536 + (u & 1) * 128;
          unsigned nf = want;
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            float4 sv[8], dv[8];
#pragma unroll
            for (int r = 0; r < 8; ++r) {
              sv[r] = sd4[(8 * h + r) * 8];
              dv[r] = pd4[(8 * h + r) * (KR_WROW / 4)];
            }
            if (h == 1 && u + 1 < U) nf = ld_acquire_s(&S.pd_flag[u + 1]);   // looked at early, needed after the additions
#pragma unroll
            for (int r = 0; r < 8; ++r) {
              acc = acc + sv[r].x * dv[r].x;   // sd_k_proj, odometer.cpp:386-391, added in the order of .sum() (:399-404)
              acc = acc + sv[r].y * dv[r].y;
              acc = acc + sv[r].z * dv[r].z;
              acc = acc + sv[r].w * dv[r].w;
            }
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&S.slot_free[u]);
          while (nf != want) nf = ld_acquire_s(&S.pd_flag[u + 1]);
        }
        const float res = kx_finish(acc);   // Eigen's redux of the eight chains
        if (!chainA) {
          if ((lane & 7) == 0 && lane < 16) S.sum[4 + (lane >> 3)] = res;
          __syncwarp();
          if (lane == 0) st_release_s(&S.b_flag, want);
        } else {
          if ((lane & 7) == 0) S.sum[lane >> 3] = res;
          float lu[36];                   // the level's LU factors (column-major), every lane alike
#pragma unroll
          for (int j = 0; j < 36; ++j) lu[j] = S.f.lu[j];
          const int lu_rank = S.f.rank;
          while (ld_acquire_s(&S.b_flag) != want) {}
          if (trace) t_c1 = clock64();
          __syncwarp();
          // 9b. solve (odometer.cpp:407, Eigen's substitution order), 10. addpose_se3, stop rule — every lane alike,
          // operands in registers
          float sumsd[6], dp[6], pr[6], Gr[12];
#pragma unroll
          for (int j = 0; j < 6; ++j) sumsd[j] = S.sum[j];
          lu6_solve_regs(lu, lu_rank, S.f.pr, S.f.qd, S.sum, S.dp);
          __syncwarp();
          const long long t_s1 = trace ? clock64() : 0;
#pragma unroll
          for (int j = 0; j < 6; ++j) { dp[j] = S.dp[j]; pr[j] = S.p[j] + dp[j]; }
          Gr[3] = Gr[7] = Gr[11] = 0.0f;
          se3_exp_f(Gr, pr);
          const long long t_s2 = trace ? clock64() : 0;
          const float normdp = ((fabsf(dp[0]) + fabsf(dp[2])) + (fabsf(dp[1]) + fabsf(dp[3]))) +
                               (fabsf(dp[4]) + fabsf(dp[5]));           // lpNorm<1>, odometer.cpp:412
          __syncwarp();
          if (lane < 6) S.p[lane] = pr[lane];
          if (lane < 12) S.G[lane] = Gr[lane];
          if (it == 0) normdp_init = normdp;
          const int cont = (it + 1 < op.maxiter) & ((normdp / normdp_init) > op.normdp_ratio);   // odometer.cpp:344-346
          nvsum += S.nv;
          if (lane == 0) {
            if (trace && trace_n < prm.trace_cap) {
              float* rec = trace + (int64_t)ICT_TRACE_FLOATS * trace_n;
              rec[0] = (float)sl;
              rec[1] = (float)it;
              for (int j = 0; j < 6; ++j) { rec[2 + j] = sumsd[j]; rec[8 + j] = dp[j]; }
              rec[14] = normdp;
              rec[15] = (float)S.nv;
              for (int j = 16; j < ICT_TRACE_FLOATS; ++j) rec[j] = 0.0f;
              rec[16] = (float)w0;
              rec[17] = (float)(t_s1 - t_c1);        // redux hand-off + solve
              if (it != 0) rec[18] = (float)(t_s2 - t_s1);   // pose update + exp
              if (it == 0) {   // first record of a level: cycles of its precompute phases
                rec[19] = (float)(lt1 - lt0);   // acquires, reference placement, window issue
                rec[20] = (float)(lt2 - lt1);   // window wait, sampling, sd store
                rec[21] = (float)(lt3 - lt2);   // Hessian
                rec[18] = (float)(lt4 - lt3);   // factorisation + first placement
              }
              rec[22] = (float)(clock64() - t_c1);   // cycles of the serial section so far (finish, solve, exp)
              rec[23] = (float)(t_c1 - t_c0);        // cycles of the chain loop
            }
            S.it = it + 1;
            S.cont[(gi + 1u) & 1u] = cont;
          }
          if (trace && trace_n < prm.trace_cap) ++trace_n;
          __syncwarp();
          if (cont) place_and_issue();   // 7. project_pt + placement for the next iteration, first windows on their way
        }
      }
      __syncthreads();
      ++it;
      ++gi;
    }
    if (chainA && lane == 0 && prm.iters) prm.iters[(int64_t)t * (op.lv_f - op.lv_l + 1) + (op.lv_f - sl)] = S.it;
  }

  if (chainA && lane == 0) {
    getpose_se3(S.p, S.G, donorm, prm.norm + 4 * (int64_t)t, prm.norm[4 * (int64_t)t + 3], prm.p_out + 6 * (int64_t)t);
    if (prm.npixres) prm.npixres[t] = (long long)nvsum * 1024;
    if (trace)
      for (int k = trace_n; k < prm.trace_cap; ++k) {
        float* rec = trace + (int64_t)ICT_TRACE_FLOATS * k;
        for (int j = 0; j < ICT_TRACE_FLOATS; ++j) rec[j] = 0.0f;
        rec[0] = -1.0f;
      }
  }
}

static int kr_pcap(const ict_optparam& op, int max_pts) { return max_pts < op.maxpttrack ? max_pts : op.maxpttrack; }

size_t kr_smem_bytes(const ict_optparam& op, int max_pts) {
  return (size_t)kr_pcap(op, max_pts) * KR_SD_BYTES_PER_POINT + KR_NSLOT * KR_SLOT_BYTES + sizeof(KrShared) + 128;
}

bool kr_supported(const ict_optparam& op, int max_pts, int tma_ok) {
  const int P = kr_pcap(op, max_pts);
  return tma_ok && op.psz == 32 && !op.dopatchnorm && P >= 1 && P <= 8 &&
         kr_smem_bytes(op, max_pts) <= (size_t)ICT_TRACK_SMEM_LIMIT;
}

template <int NPROD, int UPP>
static cudaError_t launch_track_r_t(const TrackParams& prm, size_t smem, cudaStream_t stream) {
  static bool attr_dev[64] = {};            // function attributes are per device
  int dev_ = 0;
  cudaGetDevice(&dev_);
  bool& attr_set = attr_dev[dev_ & 63];
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(k_track_r<NPROD, UPP>, cudaFuncAttributeMaxDynamicSharedMemorySize, ICT_TRACK_SMEM_LIMIT);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(k_track_r<NPROD, UPP>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  k_track_r<NPROD, UPP><<<prm.T, (NPROD + 2) * 32, smem, stream>>>(prm);
  count_launch_external();
  return cudaGetLastError();
}

cudaError_t launch_track_r(const TrackParams& prm_in, int max_pts, cudaStream_t stream) {
  if (prm_in.T <= 0) return cudaSuccess;
  TrackParams prm = prm_in;
  prm.r_pcap = kr_pcap(prm.op, max_pts);
  const size_t smem = kr_smem_bytes(prm.op, max_pts);
  if (prm.r_pcap <= 4) return launch_track_r_t<4, 2>(prm, smem, stream);
  return launch_track_r_t<8, 2>(prm, smem, stream);
}

}  // namespace ict
