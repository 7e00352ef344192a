// ict_device.cuh — device-side scalar pieces of the tracking path (sm_100a).
//
// Everything here is small, per-track (not per-pixel) arithmetic whose ORDER OF OPERATIONS follows the reference
// line by line so that the GPU result matches the reference's fp32/fp64 mix.  The translation unit is compiled
// with -fmad=false: no multiply-add is ever contracted, as in the reference's -msse4 -mavx (no -mfma) build
// (CMakeLists.txt:4).  Division and sqrt are IEEE (nvcc defaults -prec-div=true -prec-sqrt=true, no fast-math).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "ict_kernels.cuh"

#define ICT_LIEALG_SIGTHRESH 1e-4   /* utilities.h:22 */
#define ICT_LIEALG_EPSILON 1e-10    /* utilities.h:23 */

namespace ict {

// sin and cos of a double for the tracker's rotation angles.  |x| <= pi/4 (every realistic inter-frame rotation):
// the fdlibm __kernel_sin / __kernel_cos polynomials with explicit fused multiply-adds (error < 1 ulp of double,
// so the value narrowed to float equals the correctly rounded one); larger angles take the library routine.  The
// library's generic path costs several hundred dependent cycles on the one thread the whole CTA waits for.
__device__ __forceinline__ void sincos_small(double x, double* sn, double* cs) {
  if (fabs(x) > 0.78539816339744830962) {
    sincos(x, sn, cs);
    return;
  }
  const double z = x * x;
  const double S1 = -1.66666666666666324348e-01, S2 = 8.33333333332248946124e-03, S3 = -1.98412698298579493134e-04,
               S4 = 2.75573137070700676789e-06, S5 = -2.50507602534068634195e-08, S6 = 1.58969099521155010221e-10;
  const double C1 = 4.16666666666666019037e-02, C2 = -1.38888888888741095749e-03, C3 = 2.48015872894767294178e-05,
               C4 = -2.75573143513906633035e-07, C5 = 2.08757232129817482790e-09, C6 = -1.13596475577881948265e-11;
  const double v = z * x;
  const double r = __fma_rn(z, __fma_rn(z, __fma_rn(z, __fma_rn(z, S6, S5), S4), S3), S2);
  *sn = __fma_rn(v, __fma_rn(z, r, S1), x);
  const double rc = z * __fma_rn(z, __fma_rn(z, __fma_rn(z, __fma_rn(z, __fma_rn(z, C6, C5), C4), C3), C2), C1);
  const double hz = 0.5 * z;
  const double w = 1.0 - hz;
  *cs = w + (((1.0 - w) - hz) + z * rc);
}

// ---- util_SE3_coeff_to_group<T>, utilities.h:84-145 ---------------------------------------------------------
// T=float: the template's unqualified sqrt/sin/cos bind to the double C functions, so those sub-expressions are
// evaluated in double and narrowed on assignment (see oracle/ictrack_oracle.c, DEF_SE3_EXP).
template <typename T>
__device__ __forceinline__ void se3_exp(T* G, const T* p) {
  const T wx = p[3], wy = p[4], wz = p[5];
  const T xx = wx * wx, yy = wy * wy, zz = wz * wz;
  const T sig = (T)sqrt((double)(T)(xx + yy + zz));
  T sa, sb, sc;   // sin(s)/s, (1 - cos s)/s^2, (s - sin s)/s^3
  const T s2 = (sig * sig);
  const T s3 = (sig * sig * sig);
  if ((double)sig > ICT_LIEALG_SIGTHRESH) {
    double sn, cs;
    sincos_small((double)sig, &sn, &cs);
    sa = (T)(sn / (double)sig);
    sb = (T)((1 - cs) / (double)s2);
    sc = (T)(((double)sig - sn) / (double)s3);
  } else {
    sa = 1 - s2 / 6 * (1 - s2 / 20 * (1 - s2 / 42));
    sb = (T)(.5 * (double)(T)(1 - s2 / 12 * (1 - s2 / 30 * (1 - s2 / 56))));
    sc = (1 - s2 / 20 * (1 - s2 / 42 * (1 - s2 / 72))) / 6;
  }
  // rotation block R = I + sa [w]x + sb [w]x^2, entry by entry in the reference's association
  const T yyb = yy * sb, zzb = zz * sb, xxb = xx * sb;
  const T xyb = wx * wy * sb, xzb = wx * wz * sb, yzb = wy * wz * sb;
  const T xa = wx * sa, ya = wy * sa, za = wz * sa;
  G[0] = 1 - yyb - zzb;
  G[1] = xyb - za;
  G[2] = ya + xzb;
  G[4] = za + xyb;
  G[5] = 1 - xxb - zzb;
  G[6] = yzb - xa;
  G[8] = xzb - ya;
  G[9] = xa + yzb;
  G[10] = 1 - xxb - yyb;
  // translation block V u, V = I + sb [w]x + sc [w]x^2
  const T xb = wx * sb, yb = wy * sb, zb = wz * sb;
  const T xyc = wx * wy * sc, xzc = wx * wz * sc, yzc = wy * wz * sc;
  G[3] = (1 - (yy + zz) * sc) * p[0] + (xyc - zb) * p[1] + (yb + xzc) * p[2];
  G[7] = (zb + xyc) * p[0] + (1 - (xx + zz) * sc) * p[1] + (yzc - xb) * p[2];
  G[11] = (xzc - yb) * p[0] + (xb + yzc) * p[1] + (1 - (xx + yy) * sc) * p[2];
}


// The float instantiation of se3_exp with one change that cannot alter a bit: sig = sqrtf(x) instead of
// (float)sqrt((double)x).  sqrt is correctly rounded in both precisions and 53 >= 2*24 + 2, so rounding the double
// result to float equals the correctly rounded float root (no double-rounding case exists for square roots); the
// double-precision root costs ~100 dependent cycles on the thread every other warp of the CTA waits for.  Everything
// else — the double sin/cos, the three double quotients with their cancellation, the float rotation and translation
// blocks — is the reference's formula, operation by operation (utilities.h:84-145).
// ONE_LANE: called by all lanes of a converged warp with the same p; the double-precision block (sin, cos, three
// quotients: ~100 FP64 instructions, which this GPU issues at a small fraction of the FP32 rate per ACTIVE lane)
// runs on lane 0 only and its three float results are broadcast.  Same operations, same bits.
template <bool ONE_LANE = false>
__device__ __forceinline__ void se3_exp_f(float* G, const float* p) {
  const float wx = p[3], wy = p[4], wz = p[5];
  const float xx = wx * wx, yy = wy * wy, zz = wz * wz;
  const float sig = sqrtf(xx + yy + zz);
  float sa, sb, sc;   // sin(s)/s, (1 - cos s)/s^2, (s - sin s)/s^3
  const float s2 = (sig * sig);
  const float s3 = (sig * sig * sig);
  if ((double)sig > ICT_LIEALG_SIGTHRESH) {
    if (!ONE_LANE || (threadIdx.x & 31) == 0) {
      double sn, cs;
      sincos_small((double)sig, &sn, &cs);
      sa = (float)(sn / (double)sig);
      sb = (float)((1 - cs) / (double)s2);
      sc = (float)(((double)sig - sn) / (double)s3);
    } else {
      sa = sb = sc = 0.0f;
    }
    if (ONE_LANE) {
      sa = __shfl_sync(0xffffffffu, sa, 0);
      sb = __shfl_sync(0xffffffffu, sb, 0);
      sc = __shfl_sync(0xffffffffu, sc, 0);
    }
  } else {
    sa = 1 - s2 / 6 * (1 - s2 / 20 * (1 - s2 / 42));
    sb = (float)(.5 * (double)(float)(1 - s2 / 12 * (1 - s2 / 30 * (1 - s2 / 56))));
    sc = (1 - s2 / 20 * (1 - s2 / 42 * (1 - s2 / 72))) / 6;
  }
  // rotation block R = I + sa [w]x + sb [w]x^2, entry by entry in the reference's association
  const float yyb = yy * sb, zzb = zz * sb, xxb = xx * sb;
  const float xyb = wx * wy * sb, xzb = wx * wz * sb, yzb = wy * wz * sb;
  const float xa = wx * sa, ya = wy * sa, za = wz * sa;
  G[0] = 1 - yyb - zzb;
  G[1] = xyb - za;
  G[2] = ya + xzb;
  G[4] = za + xyb;
  G[5] = 1 - xxb - zzb;
  G[6] = yzb - xa;
  G[8] = xzb - ya;
  G[9] = xa + yzb;
  G[10] = 1 - xxb - yyb;
  // translation block V u, V = I + sb [w]x + sc [w]x^2
  const float xb = wx * sb, yb = wy * sb, zb = wz * sb;
  const float xyc = wx * wy * sc, xzc = wx * wz * sc, yzc = wy * wz * sc;
  G[3] = (1 - (yy + zz) * sc) * p[0] + (xyc - zb) * p[1] + (yb + xzc) * p[2];
  G[7] = (zb + xyc) * p[0] + (1 - (xx + zz) * sc) * p[1] + (yzc - xb) * p[2];
  G[11] = (xzc - yb) * p[0] + (xb + yzc) * p[1] + (1 - (xx + yy) * sc) * p[2];
}

// Production-kernel form of the float instantiation above.  sin(s)/s, (1-cos s)/s^2 and (s-sin s)/s^3 are even power
// series in s; with z = s*s formed exactly in double from the float s they are evaluated by Horner in double (ten
// terms: truncation < 1e-18 for s <= pi/4), so the three values narrowed to float equal the reference's
// double-evaluated quotients except when one of those lies within ~1e-16 relative of a float rounding boundary.
// No double division, no double sqrt (sqrtf of a float equals the double sqrt narrowed), three independent
// fused-multiply-add chains: this runs on the single thread the whole CTA waits for.
__device__ __forceinline__ void se3_exp_f32_series(float* G, const float* p) {
  const float ra1 = p[3] * p[3];
  const float ra2 = p[4] * p[4];
  const float ra3 = p[5] * p[5];
  const float sig = sqrtf(ra1 + ra2 + ra3);
  if (!((double)sig > ICT_LIEALG_SIGTHRESH) || sig > 0.78539816f) {
    se3_exp<float>(G, p);   // Taylor branch of the reference, or a rotation too large for the short series
    return;
  }
  const double z = (double)sig * (double)sig;
  // 1/(2k+1)!, 1/(2k+2)!, 1/(2k+3)! with alternating signs, k = 9 .. 0
  double a = -8.2206352466243297e-18, b = -4.1103176233121648e-19, c = -1.9572941063391263e-20;
  a = __fma_rn(a, z, 2.8114572543455206e-15);  b = __fma_rn(b, z, 1.5619206968586225e-16); c = __fma_rn(c, z, 8.2206352466243297e-18);
  a = __fma_rn(a, z, -7.6471637318198164e-13); b = __fma_rn(b, z, -4.7794773323873853e-14);  c = __fma_rn(c, z, -2.8114572543455206e-15);
  a = __fma_rn(a, z, 1.6059043836821613e-10);  b = __fma_rn(b, z, 1.1470745597729725e-11); c = __fma_rn(c, z, 7.6471637318198164e-13);
  a = __fma_rn(a, z, -2.5052108385441720e-08); b = __fma_rn(b, z, -2.0876756987868100e-09);  c = __fma_rn(c, z, -1.6059043836821613e-10);
  a = __fma_rn(a, z, 2.7557319223985893e-06);  b = __fma_rn(b, z, 2.7557319223985888e-07); c = __fma_rn(c, z, 2.5052108385441720e-08);
  a = __fma_rn(a, z, -1.9841269841269841e-04); b = __fma_rn(b, z, -2.4801587301587302e-05);  c = __fma_rn(c, z, -2.7557319223985893e-06);
  a = __fma_rn(a, z, 8.3333333333333332e-03);  b = __fma_rn(b, z, 1.3888888888888889e-03); c = __fma_rn(c, z, 1.9841269841269841e-04);
  a = __fma_rn(a, z, -1.6666666666666666e-01); b = __fma_rn(b, z, -4.1666666666666664e-02);  c = __fma_rn(c, z, -8.3333333333333332e-03);
  a = __fma_rn(a, z, 1.0);                     b = __fma_rn(b, z, 0.5);                     c = __fma_rn(c, z, 1.6666666666666666e-01);
  const float sa = (float)a, sb = (float)b, sc = (float)c;
  float tmp1 = ra2 * sb;
  float tmp2 = ra3 * sb;
  float tmp3 = ra1 * sb;
  float tmp4 = p[3] * p[4] * sb;
  float tmp5 = p[5] * sa;
  float tmp6 = p[3] * p[5] * sb;
  float tmp7 = p[4] * sa;
  float tmp8 = p[3] * sa;
  float tmp9 = p[4] * p[5] * sb;
  G[0] = 1 - tmp1 - tmp2;
  G[1] = tmp4 - tmp5;
  G[2] = tmp7 + tmp6;
  G[4] = tmp5 + tmp4;
  G[5] = 1 - tmp3 - tmp2;
  G[6] = tmp9 - tmp8;
  G[8] = tmp6 - tmp7;
  G[9] = tmp8 + tmp9;
  G[10] = 1 - tmp3 - tmp1;
  tmp1 = p[5] * sb;
  tmp2 = p[3] * p[4] * sc;
  tmp3 = p[4] * sb;
  tmp4 = p[3] * p[5] * sc;
  tmp5 = p[3] * sb;
  tmp6 = p[4] * p[5] * sc;
  G[3] = (1 - (ra2 + ra3) * sc) * p[0] + (tmp2 - tmp1) * p[1] + (tmp3 + tmp4) * p[2];
  G[7] = (tmp1 + tmp2) * p[0] + (1 - (ra1 + ra3) * sc) * p[1] + (tmp6 - tmp5) * p[2];
  G[11] = (tmp4 - tmp3) * p[0] + (tmp5 + tmp6) * p[1] + (1 - (ra1 + ra2) * sc) * p[2];
}

// ---- util_SE3_group_to_coeff<T>, utilities.h:149-241 --------------------------------------------------------
template <typename T>
__device__ __forceinline__ void se3_log(T* p, const T* G) {
  const T tr = G[0] + G[5] + G[10];
  const T theta = (T)acos((double)(T)(0.5f * (tr - 1)));
  // W = theta / (2 sin theta) (R - R^T) = [[0, a, b], [-a, 0, c], [-b, -c, 0]];  Q = W^2 (symmetric: 6 entries)
  T a = 0, b = 0, c = 0;
  T q00 = 0, q01 = 0, q02 = 0, q11 = 0, q12 = 0, q22 = 0;
  if ((double)theta < ICT_LIEALG_EPSILON) {
    p[3] = 0.0f;
    p[4] = 0.0f;
    p[5] = 0.0f;
  } else {
    const T half_over_sinc = (T)((double)theta / ((double)2.0f * sin((double)theta)));
    a = half_over_sinc * (G[1] - G[4]);
    b = half_over_sinc * (G[2] - G[8]);
    c = half_over_sinc * (G[6] - G[9]);
    p[3] = -c;
    p[4] = b;
    p[5] = -a;
    const T aa = a * a, bb = b * b, cc = c * c;
    q00 = -aa - bb;
    q01 = -b * c;
    q02 = a * c;
    q11 = -aa - cc;
    q12 = -a * b;
    q22 = -bb - cc;
  }
  T th;   // (1 - (theta/2) / tan(theta/2)) / theta^2
  if ((double)theta < ICT_LIEALG_SIGTHRESH)
    th = 1.0f / 12.0f;
  else
    th = (T)(((double)1.0f - (double)theta / ((double)2.0f * tan((double)(T)(theta / 2.0f)))) /
             (double)(T)(theta * theta));
  // u = (I - W/2 + th Q) t, row by row
  const T na = -a, nb = -b, nc = -c;
  const T v00 = 1.0f + th * q00, v01 = -0.5f * a + th * q01, v02 = -0.5f * b + th * q02;
  const T v10 = -0.5f * na + th * q01, v11 = 1.0f + th * q11, v12 = -0.5f * c + th * q12;
  const T v20 = -0.5f * nb + th * q02, v21 = -0.5f * nc + th * q12, v22 = 1.0f + th * q22;
  p[0] = v00 * G[3] + v01 * G[7] + v02 * G[11];
  p[1] = v10 * G[3] + v11 * G[7] + v12 * G[11];
  p[2] = v20 * G[3] + v21 * G[7] + v22 * G[11];
}

// ---- PoseClass::setpose_se3, pose.cpp:25-76 -------------------------------------------------------------------
static __device__ __noinline__ void setpose_se3(const double* p_in, bool donorm, const double* meanshift, double varval,
                                   float* cpos_p, float* cpos_G) {
  double p[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) p[k] = p_in[k];
  if (donorm) {
    double G[12], t[3];
    se3_exp<double>(G, p);
    t[0] = -G[0] * G[3] - G[4] * G[7] - G[8] * G[11];
    t[1] = -G[1] * G[3] - G[5] * G[7] - G[9] * G[11];
    t[2] = -G[2] * G[3] - G[6] * G[7] - G[10] * G[11];
    t[0] = (t[0] - meanshift[0]) / varval;
    t[1] = (t[1] - meanshift[1]) / varval;
    t[2] = (t[2] - meanshift[2]) / varval;
    G[3] = -G[0] * t[0] - G[1] * t[1] - G[2] * t[2];
    G[7] = -G[4] * t[0] - G[5] * t[1] - G[6] * t[2];
    G[11] = -G[8] * t[0] - G[9] * t[1] - G[10] * t[2];
    se3_log<double>(p, G);
  }
#pragma unroll
  for (int k = 0; k < 6; ++k) cpos_p[k] = (float)p[k];
  se3_exp<float>(cpos_G, cpos_p);
}

// ---- PoseClass::getPose_se3, pose.cpp:79-113 ------------------------------------------------------------------
static __device__ __noinline__ void getpose_se3(const float* cpos_p, const float* cpos_G, bool donorm, const double* meanshift,
                                   double varval, double* p_out) {
  float pu[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) pu[k] = cpos_p[k];
  if (donorm) {
    float G[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) G[k] = cpos_G[k];
    double t[3];
    t[0] = (double)(-G[0] * G[3] - G[4] * G[7] - G[8] * G[11]);   // fp32 expression widened on assignment
    t[1] = (double)(-G[1] * G[3] - G[5] * G[7] - G[9] * G[11]);
    t[2] = (double)(-G[2] * G[3] - G[6] * G[7] - G[10] * G[11]);
    t[0] = t[0] * varval + meanshift[0];
    t[1] = t[1] * varval + meanshift[1];
    t[2] = t[2] * varval + meanshift[2];
    G[3] = (float)(-(double)G[0] * t[0] - (double)G[1] * t[1] - (double)G[2] * t[2]);
    G[7] = (float)(-(double)G[4] * t[0] - (double)G[5] * t[1] - (double)G[6] * t[2]);
    G[11] = (float)(-(double)G[8] * t[0] - (double)G[9] * t[1] - (double)G[10] * t[2]);
    se3_log<float>(pu, G);
  }
#pragma unroll
  for (int k = 0; k < 6; ++k) p_out[k] = (double)pu[k];
}

// ---- the per-track bookkeeping every tracking kernel shares: what a track reads and reports (ictrack.h) -----------
// G (3 x 4, row-major) applied to a point, pose.cpp:307-397 / 400-488
template <typename T>
__device__ __forceinline__ void rigid_apply(const T* G, T X, T Y, T Z, T& x, T& y, T& z) {
  x = G[0] * X + G[1] * Y + G[2] * Z + G[3];
  y = G[4] * X + G[5] * Y + G[6] * Z + G[7];
  z = G[8] * X + G[9] * Y + G[10] * Z + G[11];
}

// the reference and new frame of track t; a sequence step adds its frame offset (K2v8's chains)
struct TrackFrames {
  const FrameDesc* ref;
  const FrameDesc* nw;
};
__device__ __forceinline__ TrackFrames track_frames(const TrackParams& prm, int t, int shift = 0) {
  const int rf = (prm.ref_frame ? prm.ref_frame[t] : prm.fixed_ref) + shift;
  const int nf = (prm.new_frame ? prm.new_frame[t] : prm.fixed_new) + shift;
  return {prm.frames + rf, prm.frames + nf};
}

// SetPose (pose.cpp:25-76) of track t from its row of p_in and its normalisation (norm: meanshift[3], varval)
__device__ __forceinline__ void track_setpose(const double* p_in, const double* norm, int t, bool donorm, float* p,
                                              float* G) {
  setpose_se3(p_in + 6 * (int64_t)t, donorm, norm + 4 * (int64_t)t, norm[4 * (int64_t)t + 3], p, G);
}

// project_pt_save_rotated (pose.cpp:400-488) of point i at the SetPose pose G: the camera-frame point into Xc/Yc/Zc
// (SAVE), and Get2DPoints() (odometer.h:30), the point at level lv_l, into pt2d_out (when set)
template <bool SAVE = true, typename I>
__device__ __forceinline__ void save_rotated_point(const TrackParams& prm, const float* G, int64_t off, int n_in, I i,
                                                   float X, float Y, float Z, float* Xc, float* Yc, float* Zc) {
  float xc, yc, zc;
  rigid_apply(G, X, Y, Z, xc, yc, zc);
  if (SAVE) {
    Xc[i] = xc;
    Yc[i] = yc;
    Zc[i] = zc;
  }
  if (prm.pt2d_out) {
    const int l = prm.op.lv_l;
    prm.pt2d_out[2 * off + i] = (xc / zc) * prm.cam.fx[l] + prm.cam.cx[l];
    prm.pt2d_out[2 * off + n_in + i] = (yc / zc) * prm.cam.fy[l] + prm.cam.cy[l];
  }
}

// lpNorm<1> of delta_p (odometer.cpp:412) in the reference's association order
__device__ __forceinline__ float normdp_l1(const float* dp) {
  return ((fabsf(dp[0]) + fabsf(dp[2])) + (fabsf(dp[1]) + fabsf(dp[3]))) + (fabsf(dp[4]) + fabsf(dp[5]));
}

// the stop rule (odometer.cpp:341-346) after `done` iterations of a level: go on while done < maxiter and the step
// norm relative to the level's first is above normdp_ratio.  A level starts at normdp = normdp_init = 1e-10:
// keep_iterating(op, 0, 1e-10f, 1e-10f).
__device__ __forceinline__ int keep_iterating(const ict_optparam& op, int done, float normdp, float normdp_init) {
  return (done < op.maxiter) & ((normdp / normdp_init) > op.normdp_ratio);
}

// track t's trace records (ICT_TRACE_FLOATS floats each), or null
__device__ __forceinline__ float* track_trace(const TrackParams& prm, int t) {
  return prm.trace ? prm.trace + (int64_t)t * prm.trace_cap * ICT_TRACE_FLOATS : nullptr;
}

// fields 0-15 of an iteration's trace record (level, iteration, J^T r, delta_p, normdp, visible points), 16-23 zeroed:
// kernels that record cycle counts there write them afterwards
__device__ __forceinline__ void trace_record(float* rec, int sl, int it, const float* jtr, const float* dp, float normdp,
                                             int nvis) {
  rec[0] = (float)sl;
  rec[1] = (float)it;
  for (int k = 0; k < 6; ++k) { rec[2 + k] = jtr[k]; rec[8 + k] = dp[k]; }
  rec[14] = normdp;
  rec[15] = (float)nvis;
  for (int k = 16; k < ICT_TRACE_FLOATS; ++k) rec[k] = 0.0f;
}

// the records from..cap-1 that no iteration filled: (-1, 0, ..., 0)
__device__ __forceinline__ void pad_trace(float* trace, int from, int cap) {
  if (!trace) return;
  for (int k = from; k < cap; ++k) {
    float* rec = trace + (int64_t)ICT_TRACE_FLOATS * k;
    for (int j = 0; j < ICT_TRACE_FLOATS; ++j) rec[j] = 0.0f;
    rec[0] = -1.0f;
  }
}

// iterations of level sl of track t, at iters[t][lv_f - sl] (when iters is set)
__device__ __forceinline__ void store_level_iters(int* iters, const ict_optparam& op, int t, int sl, int n) {
  if (iters) iters[(int64_t)t * (op.lv_f - op.lv_l + 1) + (op.lv_f - sl)] = n;
}

// the end of track t (one thread): getPose_se3 into row t of p_out, the pixel-residual count, the trace padding
__device__ __forceinline__ void finish_track(const TrackParams& prm, int t, bool donorm, const float* p, const float* G,
                                             double* p_out, long long* npixres, long long npix, float* trace,
                                             int trace_n) {
  getpose_se3(p, G, donorm, prm.norm + 4 * (int64_t)t, prm.norm[4 * (int64_t)t + 3], p_out + 6 * (int64_t)t);
  if (npixres) npixres[t] = npix;
  pad_trace(trace, trace_n, prm.trace_cap);
}

// ---- Hes.fullPivLu() (odometer.cpp:514), factor once per level; same elimination order as Eigen 3.3 ----------
struct Lu6 {
  float lu[36];   // column-major
  int rowtr[6], coltr[6];
  int rank;
  int pr[6];      // c[k] = b[pr[k]]   == the row transpositions applied in order
  int qd[6];      // x[qd[k]] = c[k]   == the column transpositions applied last-to-first
  float rdiag[6]; // 1 / U(k,k), for the production kernel's reciprocal back substitution
  int qc[6];      // x[j] = c[qc[j]] (inverse of qd), for the lane-parallel solve
};

// Eigen's full-pivoting elimination (pivot = first maximum in column-major order, the same divisions and rank-1
// updates, hence the same bits) by one warp, with lane j < 6 holding column j of the matrix in six registers.  The pivot search is a per-lane scan plus a three-step butterfly, the row swap is
// register renaming under predicates, the column swap and the broadcast of the scaled pivot column are shuffles.
// Called by all 32 lanes of one warp; Hs = the 21 unique sums in the order of ComputeHessian (odometer.cpp:430-455).
// A single-thread version cost ~26 000 SM cycles per level on a busy SM (dynamic indexing -> local memory,
// one long dependent chain) while every other warp of the CTA waits; this one ~2 000.
__device__ __forceinline__ void lu6_factor_warp(const float* Hs, Lu6& f) {
  const int lane = threadIdx.x & 31;
  const unsigned FULL = 0xffffffffu;
  float a[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    const int p = i < lane ? i : lane, q = i < lane ? lane : i;           // H(i, lane) = Hs[idx(min, max)]
    const int idx = p * 6 - (p * (p - 1)) / 2 + (q - p);
    a[i] = lane < 6 ? Hs[idx] : 0.0f;
  }
  int nonzero = 6;
  float maxpivot = 0.0f;
  int rowtr = 0, coltr = 0;   // lane k keeps transposition k
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    if (nonzero == 6) {       // uniform across the warp
      float bv = -1.0f;
      int bi = k, bl = lane;
#pragma unroll
      for (int i = k; i < 6; ++i) {
        const float v = fabsf(a[i]);
        if (v > bv) { bv = v; bi = i; }
      }
      if (lane < k || lane > 5) bv = -2.0f;
#pragma unroll
      for (int o = 4; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(FULL, bv, o);
        const int oi = __shfl_xor_sync(FULL, bi, o);
        const int ol = __shfl_xor_sync(FULL, bl, o);
        if (ov > bv || (ov == bv && ol < bl)) { bv = ov; bi = oi; bl = ol; }
      }
      const float biggest = __shfl_sync(FULL, bv, 0);
      const int pr = __shfl_sync(FULL, bi, 0), pc = __shfl_sync(FULL, bl, 0);
      if (biggest == 0.0f) {
        nonzero = k;
      } else {
        if (biggest > maxpivot) maxpivot = biggest;
        if (lane == k) { rowtr = pr; coltr = pc; }
        // rows k <-> pr (every lane, its own column)
#pragma unroll
        for (int i = k + 1; i < 6; ++i)
          if (pr == i) { const float t = a[k]; a[k] = a[i]; a[i] = t; }
        // columns k <-> pc
        const int src = lane == k ? pc : (lane == pc ? k : lane);
#pragma unroll
        for (int i = 0; i < 6; ++i) a[i] = __shfl_sync(FULL, a[i], src);
        if (k < 5) {
          if (lane == k) {
#pragma unroll
            for (int i = k + 1; i < 6; ++i) a[i] = a[i] / a[k];
          }
#pragma unroll
          for (int i = k + 1; i < 6; ++i) {
            const float l = __shfl_sync(FULL, a[i], k);
            if (lane > k && lane < 6) a[i] = a[i] - l * a[k];
          }
        }
      }
    }
    if (nonzero != 6 && lane == k && k >= nonzero) { rowtr = k; coltr = k; }
  }
  // diagonal, rank, reciprocals
  float diag = 0.0f;
#pragma unroll
  for (int i = 0; i < 6; ++i)
    if (lane == i) diag = a[i];
  const float premult = fabsf(maxpivot) * (1.1920929e-07f * 6.0f);
  const unsigned ok = __ballot_sync(FULL, lane < nonzero && fabsf(diag) > premult);
  // index tables of the solve: pr = the row transpositions applied in order to the identity, qc = the column
  // transpositions applied last-to-first; lane j carries entry j, transposition k comes from lane k
  int pr = lane, qc = lane;
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    const int r = __shfl_sync(FULL, rowtr, k);
    const int vk = __shfl_sync(FULL, pr, k), vr = __shfl_sync(FULL, pr, r);
    if (lane == k) pr = vr; else if (lane == r) pr = vk;
  }
#pragma unroll
  for (int k = 5; k >= 0; --k) {
    const int c = __shfl_sync(FULL, coltr, k);
    const int vk = __shfl_sync(FULL, qc, k), vc = __shfl_sync(FULL, qc, c);
    if (lane == k) qc = vc; else if (lane == c) qc = vk;
  }
  if (lane < 6) {
#pragma unroll
    for (int i = 0; i < 6; ++i) f.lu[i + 6 * lane] = a[i];
    f.rowtr[lane] = rowtr;
    f.coltr[lane] = coltr;
    f.rdiag[lane] = 1.0f / diag;
    f.pr[lane] = pr;
    f.qd[qc] = lane;
    f.qc[lane] = qc;
  }
  if (lane == 0) f.rank = __popc(ok);
  __syncwarp();
}

static __device__ __noinline__ void lu6_solve(const Lu6& f, const float* b, float* x) {
#define LU(i, j) f.lu[(i) + 6 * (j)]
  if (f.rank == 0) {
    for (int i = 0; i < 6; ++i) x[i] = 0.0f;
    return;
  }
  float c[6];
  for (int i = 0; i < 6; ++i) c[i] = b[i];
  for (int k = 0; k < 6; ++k)
    if (f.rowtr[k] != k) { float t = c[k]; c[k] = c[f.rowtr[k]]; c[f.rowtr[k]] = t; }
  for (int i = 0; i < 6; ++i)
    for (int r = i + 1; r < 6; ++r) c[r] = c[r] - c[i] * LU(r, i);
  for (int i = f.rank - 1; i >= 0; --i) {
    c[i] = c[i] / LU(i, i);
    for (int r = 0; r < i; ++r) c[r] = c[r] - c[i] * LU(r, i);
  }
  for (int i = f.rank; i < 6; ++i) c[i] = 0.0f;
  for (int k = 5; k >= 0; --k)
    if (f.coltr[k] != k) { float t = c[k]; c[k] = c[f.coltr[k]]; c[f.coltr[k]] = t; }
  for (int i = 0; i < 6; ++i) x[i] = c[i];
#undef LU
}

// FullPivLU::solve (odometer.cpp:514) as straight-line code for any rank: lu6_solve of ict_device.cuh (c = P b,
// unit-lower forward substitution over all six rows, upper backward substitution on the leading rank x rank block
// with true divisions, zeros beyond the rank, x = Q c) with the permutations folded into the index tables and the
// rank test as predicates — the same operations in the same order, hence the same bits; about 100 instructions
// instead of the loops over run-time bounds and the local-memory array of the generic routine (37 % of the 4-point
// benchmark tracks' level Hessians are rank-deficient by Eigen's threshold, so that path is not rare).
__device__ __forceinline__ void lu6_solve_exact(const Lu6& f, const float* b, float* x) {
#define LU(i, j) f.lu[(i) + 6 * (j)]
  const int rank = f.rank;
  float c0 = b[f.pr[0]], c1 = b[f.pr[1]], c2 = b[f.pr[2]], c3 = b[f.pr[3]], c4 = b[f.pr[4]], c5 = b[f.pr[5]];
  if (rank == 0) c0 = c1 = c2 = c3 = c4 = c5 = 0.0f;
  c1 = c1 - c0 * LU(1, 0); c2 = c2 - c0 * LU(2, 0); c3 = c3 - c0 * LU(3, 0); c4 = c4 - c0 * LU(4, 0); c5 = c5 - c0 * LU(5, 0);
  c2 = c2 - c1 * LU(2, 1); c3 = c3 - c1 * LU(3, 1); c4 = c4 - c1 * LU(4, 1); c5 = c5 - c1 * LU(5, 1);
  c3 = c3 - c2 * LU(3, 2); c4 = c4 - c2 * LU(4, 2); c5 = c5 - c2 * LU(5, 2);
  c4 = c4 - c3 * LU(4, 3); c5 = c5 - c3 * LU(5, 3);
  c5 = c5 - c4 * LU(5, 4);
  if (rank > 5) {
    c5 = c5 / LU(5, 5);
    c0 = c0 - c5 * LU(0, 5); c1 = c1 - c5 * LU(1, 5); c2 = c2 - c5 * LU(2, 5); c3 = c3 - c5 * LU(3, 5); c4 = c4 - c5 * LU(4, 5);
  } else c5 = 0.0f;
  if (rank > 4) {
    c4 = c4 / LU(4, 4);
    c0 = c0 - c4 * LU(0, 4); c1 = c1 - c4 * LU(1, 4); c2 = c2 - c4 * LU(2, 4); c3 = c3 - c4 * LU(3, 4);
  } else c4 = 0.0f;
  if (rank > 3) {
    c3 = c3 / LU(3, 3);
    c0 = c0 - c3 * LU(0, 3); c1 = c1 - c3 * LU(1, 3); c2 = c2 - c3 * LU(2, 3);
  } else c3 = 0.0f;
  if (rank > 2) {
    c2 = c2 / LU(2, 2);
    c0 = c0 - c2 * LU(0, 2); c1 = c1 - c2 * LU(1, 2);
  } else c2 = 0.0f;
  if (rank > 1) {
    c1 = c1 / LU(1, 1);
    c0 = c0 - c1 * LU(0, 1);
  } else c1 = 0.0f;
  c0 = rank > 0 ? c0 / LU(0, 0) : 0.0f;
  x[f.qd[0]] = c0; x[f.qd[1]] = c1; x[f.qd[2]] = c2; x[f.qd[3]] = c3; x[f.qd[4]] = c4; x[f.qd[5]] = c5;
#undef LU
}


// lu6_solve_exact with the factors in registers (lu: column-major, uniform across the calling lanes) and the two
// permutations applied through shared memory (b and x live there): same operations, same order, same bits.
__device__ __forceinline__ void lu6_solve_regs(const float* lu, int rank, const int* pr, const int* qd, const float* b, float* x) {
#define LU(i, j) lu[(i) + 6 * (j)]
  float c0 = b[pr[0]], c1 = b[pr[1]], c2 = b[pr[2]], c3 = b[pr[3]], c4 = b[pr[4]], c5 = b[pr[5]];
  if (rank == 0) c0 = c1 = c2 = c3 = c4 = c5 = 0.0f;
  c1 = c1 - c0 * LU(1, 0); c2 = c2 - c0 * LU(2, 0); c3 = c3 - c0 * LU(3, 0); c4 = c4 - c0 * LU(4, 0); c5 = c5 - c0 * LU(5, 0);
  c2 = c2 - c1 * LU(2, 1); c3 = c3 - c1 * LU(3, 1); c4 = c4 - c1 * LU(4, 1); c5 = c5 - c1 * LU(5, 1);
  c3 = c3 - c2 * LU(3, 2); c4 = c4 - c2 * LU(4, 2); c5 = c5 - c2 * LU(5, 2);
  c4 = c4 - c3 * LU(4, 3); c5 = c5 - c3 * LU(5, 3);
  c5 = c5 - c4 * LU(5, 4);
  if (rank > 5) {
    c5 = c5 / LU(5, 5);
    c0 = c0 - c5 * LU(0, 5); c1 = c1 - c5 * LU(1, 5); c2 = c2 - c5 * LU(2, 5); c3 = c3 - c5 * LU(3, 5); c4 = c4 - c5 * LU(4, 5);
  } else c5 = 0.0f;
  if (rank > 4) {
    c4 = c4 / LU(4, 4);
    c0 = c0 - c4 * LU(0, 4); c1 = c1 - c4 * LU(1, 4); c2 = c2 - c4 * LU(2, 4); c3 = c3 - c4 * LU(3, 4);
  } else c4 = 0.0f;
  if (rank > 3) {
    c3 = c3 / LU(3, 3);
    c0 = c0 - c3 * LU(0, 3); c1 = c1 - c3 * LU(1, 3); c2 = c2 - c3 * LU(2, 3);
  } else c3 = 0.0f;
  if (rank > 2) {
    c2 = c2 / LU(2, 2);
    c0 = c0 - c2 * LU(0, 2); c1 = c1 - c2 * LU(1, 2);
  } else c2 = 0.0f;
  if (rank > 1) {
    c1 = c1 / LU(1, 1);
    c0 = c0 - c1 * LU(0, 1);
  } else c1 = 0.0f;
  c0 = rank > 0 ? c0 / LU(0, 0) : 0.0f;
  __syncwarp();
  x[qd[0]] = c0; x[qd[1]] = c1; x[qd[2]] = c2; x[qd[3]] = c3; x[qd[4]] = c4; x[qd[5]] = c5;
#undef LU
}

// The full-rank solve of the fast-mode kernels, spread over six lanes (called by a full warp, rank 6): lane r carries
// c_r; one shuffle per elimination step broadcasts the pivot row's value.  Forward and backward substitution in
// lu6_solve's order, but the six divisions by the pivots are multiplications by their (correctly rounded, once per
// level) reciprocals: at most one ulp per division from the reference's x / u — far below what the fp32 right-hand
// side carries — and no ~10-deep dependent division chains in the code the whole CTA waits for.  About 50 issued
// instructions instead of 130 for the straight-line single-lane form.  Returns x_lane (valid in lanes 0..5).
__device__ __forceinline__ float lu6_solve_warp_rcp(const Lu6& f, const float* b) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31, r = lane < 6 ? lane : 0;
  float c = b[f.pr[r]];
  float m[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) m[i] = f.lu[r + 6 * i];     // row r of L\U
  const float rd = f.rdiag[r];
  const int qc = f.qc[r];
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    const float ci = __shfl_sync(FULL, c, i);
    if (r > i) c = c - ci * m[i];
  }
#pragma unroll
  for (int i = 5; i >= 0; --i) {
    if (r == i) c = c * rd;
    const float ci = __shfl_sync(FULL, c, i);
    if (r < i) c = c - ci * m[i];
  }
  return __shfl_sync(FULL, c, qc);
}

// ---- bilinear patch placement, util_getPatch / util_getPatch_grad (utilities.cpp:65-94, 127-157) -----------------
// For a patch centre `mid` returns the flat offset of the patch's first pixel (row pos1+pszd2, col pos0+pszd2 of
// the padded plane) and the four constant weights.
struct PatchPlace {
  int base;
  float w0, w1, w2, w3;
};
// consistent == true (ICT_ROBUST_FLOOR, opt-in, not parity): the patch origin is floor(x) + 1 for every x, instead of the
// reference's ceil(x + 1e-5f), which equals floor(x) for integer x >= 256 and floor(x) + 2 for frac(x) > 1 - 1e-5
// (SURVEY.md §9.2): template and new-frame patches are then sampled on the same grid wherever their centres fall.
__device__ __forceinline__ PatchPlace patch_place(float mx, float my, int pszd2, int width, bool consistent = false) {
  PatchPlace q;
  const int pos2 = (int)floorf(mx);
  const int pos3 = (int)floorf(my);
  const int pos0 = consistent ? pos2 + 1 : (int)ceilf(mx + .00001f);
  const int pos1 = consistent ? pos3 + 1 : (int)ceilf(my + .00001f);
  const float r0 = mx - (float)pos2;
  const float r1 = my - (float)pos3;
  q.w0 = r0 * r1;
  q.w1 = (1 - r0) * r1;
  q.w2 = r0 * (1 - r1);
  q.w3 = (1 - r0) * (1 - r1);
  q.base = (pos1 + pszd2) * width + pos0 + pszd2;
  return q;
}

// we[0]*a + we[1]*b + we[2]*c + we[3]*d, left to right (utilities.cpp:107,181-183)
__device__ __forceinline__ float bilin4(const float* __restrict__ img, int addr, int width, float w0, float w1,
                                        float w2, float w3) {
  const float a = __ldg(img + addr);
  const float b = __ldg(img + addr - 1);
  const float c = __ldg(img + addr - width);
  const float d = __ldg(img + addr - width - 1);
  return ((w0 * a + w1 * b) + w2 * c) + w3 * d;
}

// ---- per-point steepest-descent coefficients, odometer.cpp:306-326 ---------------------------------------------
// sd1 = dx*c[0]; sd2 = dy*c[1]; sd3 = dx*c[2]+dy*c[3]; sd4 = dx*c[4]+dy*c[5]; sd5 = dx*c[6]+dy*c[7];
// sd6 = dx*c[8]+dy*c[9].  The two "1.0 + ..." terms are double in the reference and narrowed by Eigen's scalar op.
__device__ __forceinline__ void sd_coefs(float pt_x, float pt_y, float pt_z, float fx, float fy, float* c) {
  const float pt_zsq = pt_z * pt_z;
  c[0] = (fx / pt_z);
  c[1] = (fy / pt_z);
  c[2] = (-pt_x / pt_zsq * fx);
  c[3] = (-pt_y / pt_zsq * fy);
  c[4] = (-pt_x * pt_y / pt_zsq * fx);
  c[5] = (float)((-(1.0 + (double)(pt_y * pt_y / pt_zsq))) * (double)fy);
  c[6] = (float)((1.0 + (double)(pt_x * pt_x / pt_zsq)) * (double)fx);
  c[7] = (pt_x * pt_y / pt_zsq * fy);
  c[8] = (-pt_y / pt_z * fx);
  c[9] = (pt_x / pt_z * fy);
}

__device__ __forceinline__ void sd_values(float gx, float gy, const float* c, float* sd) {
  sd[0] = gx * c[0];
  sd[1] = gy * c[1];
  sd[2] = gx * c[2] + gy * c[3];
  sd[3] = gx * c[4] + gy * c[5];
  sd[4] = gx * c[6] + gy * c[7];
  sd[5] = gx * c[8] + gy * c[9];
}

// The six steepest-descent values of a pixel are sd_k = dx*A_k + dy*B_k with (A_k, B_k) constant per POINT
// (odometer.cpp:317-326).  The production kernel therefore never forms them per pixel: per point it accumulates
//   J^T r :  ax = sum dx*pdiff, ay = sum dy*pdiff            ->  sum_k += A_k*ax + B_k*ay
//   Hessian: sxx = sum dx*dx, sxy = sum dx*dy, syy = sum dy*dy -> H_ab += A_a A_b sxx + (A_a B_b + B_a A_b) sxy + B_a B_b syy
// which is the reference's sum with the distributive law applied (exact in real arithmetic; in fp32 it moves the
// result by the same ~1e-7 relative as a different summation order does) and cuts the per-pixel arithmetic of the
// iteration from 34 to 12 flops and of the Hessian from 56 to 6.  The general kernel k_track keeps the per-pixel
// form and is bit-identical to the reference in sum_mode 1.
__device__ __forceinline__ void fold_jtr(float* acc, const float* cf, float ax, float ay) {
  acc[0] = acc[0] + ax * cf[0];
  acc[1] = acc[1] + ay * cf[1];
  acc[2] = acc[2] + (ax * cf[2] + ay * cf[3]);
  acc[3] = acc[3] + (ax * cf[4] + ay * cf[5]);
  acc[4] = acc[4] + (ax * cf[6] + ay * cf[7]);
  acc[5] = acc[5] + (ax * cf[8] + ay * cf[9]);
}

__device__ __forceinline__ void fold_hessian(float* acc, const float* cf, float sxx, float sxy, float syy) {
  const float A[6] = {cf[0], 0.0f, cf[2], cf[4], cf[6], cf[8]};
  const float B[6] = {0.0f, cf[1], cf[3], cf[5], cf[7], cf[9]};
  int k = 0;
#pragma unroll
  for (int a = 0; a < 6; ++a)
#pragma unroll
    for (int b = a; b < 6; ++b) {
      acc[k] = acc[k] + ((A[a] * A[b]) * sxx + (A[a] * B[b] + B[a] * A[b]) * sxy + (B[a] * B[b]) * syy);
      ++k;
    }
}

// deterministic warp tree (fixed order, no atomics on floats)
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = v + __shfl_down_sync(0xffffffffu, v, o);
  return v;
}

// ---- reference-order reductions (Eigen's vectorised .sum(), W-float packets, two accumulators) -------------------
// W = 4 (SSE Packet4f, Eigen 3.3 built without AVX): eight interleaved SEQUENTIAL fp32 chains; W = 8 (AVX Packet8f):
// sixteen.  Chain c adds v[c], v[2W+c], ... ; then p0+p1, one odd packet, for W = 8 predux4(lo + hi), predux
// (a0+a2)+(a1+a3), scalar tail — see oracle/ictrack_oracle.c DEF_PACKET_SUM and ict_kernels.cu (sum_mode 1).
// chain c (< 2W) of the two-accumulator body: sum over e = c, c+2W, ... < as2 (values beyond `valid` are zeros)
template <int W, typename F>
__device__ __forceinline__ float eigen_chain(F v, int c, int as2, int valid) {
  if (c >= as2) return 0.0f;
  float s = c < valid ? v(c) : 0.0f;
  const int lim = as2 < valid ? as2 : valid;
  for (int e = c + 2 * W; e < lim; e += 2 * W) s = s + v(e);
  return s;
}
// combine the 2W chains + the odd packet + the scalar tail exactly like redux_impl::run
template <int W, typename F>
__device__ __forceinline__ float eigen_finish(const float* ch, F v, int N, int valid) {
  static_assert(W == 4 || W == 8, "Eigen float packets are 4 (SSE) or 8 (AVX) wide");
  const int as1 = (N / W) * W, as2 = (N / (2 * W)) * (2 * W);
  auto val = [&](int e) { return e < valid ? v(e) : 0.0f; };
  float res;
  if (N == 0) return 0.0f;
  if (as1) {
    float p0[W];
    if (as1 > W) {
      for (int j = 0; j < W; ++j) p0[j] = ch[j] + ch[W + j];
      if (as1 > as2)
        for (int j = 0; j < W; ++j) p0[j] = p0[j] + val(as2 + j);
    } else {
      for (int j = 0; j < W; ++j) p0[j] = val(j);
    }
    if (W == 8)                                       // predux<Packet8f> = predux(lo + hi)
      for (int j = 0; j < 4; ++j) p0[j] = p0[j] + p0[j + 4];
    res = (p0[0] + p0[2]) + (p0[1] + p0[3]);
    for (int e = as1; e < N; ++e) res = res + val(e);
  } else {
    res = val(0);
    for (int e = 1; e < N; ++e) res = res + val(e);
  }
  return res;
}
// whole sum by ONE thread (patch means: N = psz*psz)
template <int W, typename F>
__device__ __forceinline__ float eigen_sum_serial(F v, int N) {
  float ch[2 * W];
  const int as2 = (N / (2 * W)) * (2 * W);
  for (int c = 0; c < 2 * W; ++c) ch[c] = eigen_chain<W>(v, c, as2, N);
  return eigen_finish<W>(ch, v, N, N);
}



// Sums NV (<= 24) per-thread values over the 32 lanes of a warp with a "halving" butterfly: at each step a lane keeps
// one half of its values, sends the other half to its partner and adds what it receives, so the number of live values
// halves together with the number of lanes that still hold distinct partial sums (27 shuffles for 21 values, 15 for
// 6, instead of 5 per value).  Fixed order => deterministic.  On return lane L < 32 holds, in out, the total of
// value index slot_of(L); with NV <= 24 the totals sit in lanes 0,4,8,..: value k in lane (k % 8) * 4 (+ k / 8 picks
// which of the up to three results the lane holds).  Callers use warp_sum_store below.
template <int NV>
__device__ __forceinline__ void warp_sum_store(const float* acc, float* dst /* NV floats, shared */) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  float v[24];
#pragma unroll
  for (int k = 0; k < 24; ++k) v[k] = k < NV ? acc[k] : 0.0f;
  // offset 16: 24 -> 12
  {
    const bool up = (lane & 16) != 0;
#pragma unroll
    for (int j = 0; j < 12; ++j) {
      const float send = up ? v[j] : v[j + 12], keep = up ? v[j + 12] : v[j];
      v[j] = keep + __shfl_xor_sync(FULL, send, 16);
    }
  }
  // offset 8: 12 -> 6
  {
    const bool up = (lane & 8) != 0;
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      const float send = up ? v[j] : v[j + 6], keep = up ? v[j + 6] : v[j];
      v[j] = keep + __shfl_xor_sync(FULL, send, 8);
    }
  }
  // offset 4: 6 -> 3
  {
    const bool up = (lane & 4) != 0;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const float send = up ? v[j] : v[j + 3], keep = up ? v[j + 3] : v[j];
      v[j] = keep + __shfl_xor_sync(FULL, send, 4);
    }
  }
  // offsets 2, 1: plain butterfly on the three remaining values
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    v[j] = v[j] + __shfl_xor_sync(FULL, v[j], 2);
    v[j] = v[j] + __shfl_xor_sync(FULL, v[j], 1);
  }
  // lane with bits (16,8,4) = (a,b,c) holds values 12a + 6b + 3c + {0,1,2}
  if ((lane & 3) == 0) {
    const int base = ((lane >> 4) & 1) * 12 + ((lane >> 3) & 1) * 6 + ((lane >> 2) & 1) * 3;
#pragma unroll
    for (int j = 0; j < 3; ++j)
      if (base + j < NV) dst[base + j] = v[j];
  }
}

// Six values: one halving step (6 -> 3), then a plain butterfly: 15 shuffles instead of 30.
__device__ __forceinline__ void warp_sum6_store(const float* acc, float* dst /* 6 floats, shared */) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31;
  const bool up = (lane & 16) != 0;
  float v[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const float send = up ? acc[j] : acc[j + 3], keep = up ? acc[j + 3] : acc[j];
    v[j] = keep + __shfl_xor_sync(FULL, send, 16);
  }
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    v[j] = v[j] + __shfl_xor_sync(FULL, v[j], 8);
    v[j] = v[j] + __shfl_xor_sync(FULL, v[j], 4);
    v[j] = v[j] + __shfl_xor_sync(FULL, v[j], 2);
    v[j] = v[j] + __shfl_xor_sync(FULL, v[j], 1);
  }
  if ((lane & 15) == 0) {
    const int base = up ? 3 : 0;
#pragma unroll
    for (int j = 0; j < 3; ++j) dst[base + j] = v[j];
  }
}

// ---- shared-memory barriers (mbarrier) and bulk asynchronous copies (sm_90+ PTX) ----------------------------------------
__device__ __forceinline__ unsigned ict_saddr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* b, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(ict_saddr(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* b) {   // release at CTA scope
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(ict_saddr(b)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* b, unsigned parity) {   // acquire at CTA scope
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "KX_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra KX_DONE;\n"
      "bra KX_WAIT;\n"
      "KX_DONE:\n"
      "}\n" ::"r"(ict_saddr(b)), "r"(parity)
      : "memory");
}

// producer side of a bulk copy: the barrier's phase completes when `bytes` have landed (and the one arrival is in)
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* b, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(ict_saddr(b)), "r"(bytes) : "memory");
}
// global -> shared bulk copy through the copy engine of the SM (TMA, non-tensor form): 16-byte aligned addresses,
// size a multiple of 16; completion is signalled on the mbarrier
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* b) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   ict_saddr(dst)),
               "l"(src), "r"(bytes), "r"(ict_saddr(b))
               : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

}  // namespace ict
