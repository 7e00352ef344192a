// ict_kernel_v2.cuh — device helpers shared by the float4-row-quad kernels for 32x32 patches:
// K2v2 (ict_kernel_v2.cu, production), K2v8 (ict_kernel_v8.cu, 8x8 patches) and K2x (ict_kernel_x.cu,
// reference-order sums): placement, template gather, the per-level solve matrix, the register-resident exp.
#pragma once
#include "ict_device.cuh"

namespace ict {

__device__ __forceinline__ float4 ld4s(const float* p) { return *reinterpret_cast<const float4*>(p); }

// project_pt (pose.cpp:307-397) of one point at level intrinsics (fx, fy, cx, cy) + util_getPatch placement
// (utilities.cpp:65-94): the reference's operation order, no fused operations.  Writes {base, vis, -, -}, {w0..w3}.
__device__ __forceinline__ int place_point(const float* G, float X, float Y, float Z, float fx, float fy, float cx,
                                           float cy, float swo, float sho, int width, float4* dst, int pszd2 = 16,
                                           bool consistent = false) {
  float tx, ty, tz;
  rigid_apply(G, X, Y, Z, tx, ty, tz);
  const float mx = (tx / tz) * fx + cx, my = (ty / tz) * fy + cy;
  const int vis = (mx >= 0) & (my >= 0) & (mx <= swo) & (my <= sho);   // odometer.cpp:369-371 (NaN -> outside)
  PatchPlace pl = {0, 0.f, 0.f, 0.f, 0.f};
  if (vis) pl = patch_place(mx, my, pszd2, width, consistent);
  dst[0] = make_float4(__int_as_float(pl.base), __int_as_float(vis), 0.0f, 0.0f);
  dst[1] = make_float4(pl.w0, pl.w1, pl.w2, pl.w3);
  return vis;
}

// util_getPatch_grad (utilities.cpp:160-185) for KT consecutive rows of one patch column: p points at the row ABOVE
// the first one (the bilinear sample of row r reads rows r and r-1, columns c and c-1); unfused, in the reference's
// order ((w0*a + w1*b) + w2*c) + w3*d.  Writes KT/4 float4 row-quads at dst, dst + 32, ...
template <int KT>
__device__ __forceinline__ void gather_plane(const float* __restrict__ p, int width, const float4 w, float4* dst) {
  float a[KT + 1], b[KT + 1];
#pragma unroll
  for (int j = 0; j <= KT; ++j) {
    a[j] = __ldg(p + j * width);
    b[j] = __ldg(p + j * width - 1);
  }
#pragma unroll
  for (int jq = 0; jq < KT / 4; ++jq) {
    float r[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int row = 4 * jq + j + 1;
      r[j] = ((w.x * a[row] + w.y * b[row]) + w.z * a[row - 1]) + w.w * b[row - 1];
    }
    dst[jq * 32] = make_float4(r[0], r[1], r[2], r[3]);
  }
}

struct __align__(16) V2Shared {
  float Hinv[64];          // rows of M (delta_p = M * J^T r; H^-1 at full rank), 8 floats per row, rows/columns 6, 7 zero
  float G[12];
  float p[8];
  float Hsum[24];
  float lvl_cycles, gather_cycles;
  float Ex[12], dps[8];    // robustness mode "compose": exp(delta_p) and delta_p of the running iteration
  int cont, it;
};

// The matrix M with delta_p = M * b, b = J^T r, that Eigen's FullPivLU::solve applies (odometer.cpp:514): c = P b,
// unit-lower forward substitution, upper backward substitution on the leading rank x rank block only, the other
// unknowns zero, x = Q c.  For rank 6 M is H^-1; for a rank-deficient Hessian it is Eigen's truncated solve — linear
// in b either way, so it is tabulated once per level, from the Hessian directly, without a factorisation: symmetric
// Gauss-Jordan sweeps with the pivot taken as the largest remaining diagonal entry.  For a symmetric positive semi-definite matrix that is the pivot
// Eigen's full pivoting finds (|a_ij| <= max(a_ii, a_jj)), the Schur complements that appear are the ones its
// elimination forms, and stopping at the first pivot <= maxpivot * 6 eps is its rank rule (FullPivLU::rank with the
// default threshold): after sweeping the index set K the K x K block holds -(H_KK)^-1, which is what the truncated
// solve applies to b_K, and the unknowns outside K are zero.
// Lane q < 21 holds H(i, j), i <= j, q = the position in ComputeHessian's order (row-major upper triangle).  Per
// sweep: one integer REDUX + vote for the pivot (positive floats order like their bit patterns), one IEEE
// reciprocal, two shuffles for a_ik and a_kj, one update — ~35 instructions, all lanes, six sweeps at most.
__device__ __forceinline__ void sweep6_solve_matrix(float a, float* Hinv /* shared, 8 x 8, zeroed */) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  int i = 0, j = 0;
  {
    int k = lane < 21 ? lane : 0, len = 6;
    while (k >= len) { k -= len; --len; ++i; }
    j = i + k;
  }
  // source lanes of a_ik and a_kj for k = 0..5, five bits each
  unsigned tu = 0, tv = 0;
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    const int iu = min(i, k), ju = max(i, k), iv = min(j, k), jv = max(j, k);
    tu |= (unsigned)(iu * 6 - (iu * (iu - 1)) / 2 + (ju - iu)) << (5 * k);
    tv |= (unsigned)(iv * 6 - (iv * (iv - 1)) / 2 + (jv - iv)) << (5 * k);
  }
  const bool diag = (i == j) && lane < 21;
  unsigned done = 0;                     // swept indices (uniform)
  float maxpivot = 0.0f;
#pragma unroll 1
  for (int step = 0; step < 6; ++step) {
    const unsigned bits = (diag && !((done >> i) & 1u) && a > 0.0f) ? __float_as_uint(a) : 0u;
    const unsigned best = __reduce_max_sync(FULL, bits);
    const float pivot = __uint_as_float(best);
    if (step == 0) maxpivot = pivot;
    if (!(pivot > maxpivot * (1.1920929e-07f * 6.0f))) break;   // rank reached (or H == 0)
    const int src = __ffs(__ballot_sync(FULL, bits == best)) - 1;
    const int k = __shfl_sync(FULL, i, src);
    const float r = 1.0f / pivot;
    const float u = __shfl_sync(FULL, a, (tu >> (5 * k)) & 31u);   // a_ik
    const float v = __shfl_sync(FULL, a, (tv >> (5 * k)) & 31u);   // a_kj
    if (i == k && j == k) a = -r;
    else if (i == k || j == k) a = a * r;
    else a = a - (u * r) * v;
    done |= 1u << k;
  }
  if (lane < 21) {
    const float m = (((done >> i) & 1u) && ((done >> j) & 1u)) ? -a : 0.0f;
    Hinv[i * 8 + j] = m;
    Hinv[j * 8 + i] = m;
  }
}

// the reference's float exp for the two rare branches (Taylor for sigma <= 1e-4, library sincos beyond pi/4)
static __device__ __noinline__ void se3_exp_rare(float* G, const float* p) { se3_exp<float>(G, p); }

// util_SE3_coeff_to_group<float> (utilities.h:84-145) on register operands, every lane of the serial warp alike.
// sa = sin(s)/s, sb = (1-cos s)/s^2, sc = (s-sin s)/s^3 are even power series in z = s*s = |omega|^2; for
// 1e-8 < z <= (pi/4)^2 they are evaluated by a six-term fused Horner scheme in fp32 directly from z (truncation
// < 1e-11; the result is within one float ulp of the reference's double-evaluated quotient narrowed to float, and
// needs neither the square root nor double arithmetic on the critical path of the iteration).  Outside that range
// (the reference's Taylor branch below sigma = 1e-4, or a rotation beyond 45 degrees per pose) the reference's
// own formula runs.  The rotation and translation blocks follow the reference's unfused operation order.
// sG / sp: shared-memory copies of G and p (sp already holds the new coefficients) for the rare branch, which one
// lane runs through the noinline reference formula so that G itself never has its address taken (registers).
__device__ __forceinline__ void se3_exp_regs(float* G, float p0, float p1, float p2, float p3, float p4, float p5,
                                             float* sG, const float* sp) {
  const float ra1 = p3 * p3, ra2 = p4 * p4, ra3 = p5 * p5;
  const float z = ra1 + ra2 + ra3;
  if (!(z > 1.0000001e-8f) || z > 0.61685f) {   // uniform across the warp
    __syncwarp();
    if ((threadIdx.x & 31) == 0) se3_exp_rare(sG, sp);
    __syncwarp();
#pragma unroll
    for (int k = 0; k < 12; ++k) G[k] = sG[k];
    return;
  }
  float sa = -2.5052108385441720e-08f, sb = -2.0876756987868100e-09f, sc = -1.6059043836821613e-10f;
  sa = fmaf(sa, z, 2.7557319223985893e-06f);  sb = fmaf(sb, z, 2.7557319223985888e-07f);  sc = fmaf(sc, z, 2.5052108385441720e-08f);
  sa = fmaf(sa, z, -1.9841269841269841e-04f); sb = fmaf(sb, z, -2.4801587301587302e-05f); sc = fmaf(sc, z, -2.7557319223985893e-06f);
  sa = fmaf(sa, z, 8.3333333333333332e-03f);  sb = fmaf(sb, z, 1.3888888888888889e-03f);  sc = fmaf(sc, z, 1.9841269841269841e-04f);
  sa = fmaf(sa, z, -1.6666666666666666e-01f); sb = fmaf(sb, z, -4.1666666666666664e-02f); sc = fmaf(sc, z, -8.3333333333333332e-03f);
  sa = fmaf(sa, z, 1.0f);                     sb = fmaf(sb, z, 0.5f);                     sc = fmaf(sc, z, 1.6666666666666666e-01f);
  float tmp1 = ra2 * sb;
  float tmp2 = ra3 * sb;
  float tmp3 = ra1 * sb;
  float tmp4 = p3 * p4 * sb;
  float tmp5 = p5 * sa;
  float tmp6 = p3 * p5 * sb;
  float tmp7 = p4 * sa;
  float tmp8 = p3 * sa;
  float tmp9 = p4 * p5 * sb;
  G[0] = 1 - tmp1 - tmp2;
  G[1] = tmp4 - tmp5;
  G[2] = tmp7 + tmp6;
  G[4] = tmp5 + tmp4;
  G[5] = 1 - tmp3 - tmp2;
  G[6] = tmp9 - tmp8;
  G[8] = tmp6 - tmp7;
  G[9] = tmp8 + tmp9;
  G[10] = 1 - tmp3 - tmp1;
  tmp1 = p5 * sb;
  tmp2 = p3 * p4 * sc;
  tmp3 = p4 * sb;
  tmp4 = p3 * p5 * sc;
  tmp5 = p3 * sb;
  tmp6 = p4 * p5 * sc;
  G[3] = (1 - (ra2 + ra3) * sc) * p0 + (tmp2 - tmp1) * p1 + (tmp3 + tmp4) * p2;
  G[7] = (tmp1 + tmp2) * p0 + (1 - (ra1 + ra3) * sc) * p1 + (tmp6 - tmp5) * p2;
  G[11] = (tmp4 - tmp3) * p0 + (tmp5 + tmp6) * p1 + (1 - (ra1 + ra2) * sc) * p2;
}

}  // namespace ict
