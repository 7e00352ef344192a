/*
 * ictrack_oracle.c — CPU ORACLE (test infrastructure, NOT the product; see ictrack_oracle.h).
 *
 * Restates, function by function, the reference's tracking path.  Every function names the
 * reference file:line it follows.  Build with the reference's release flags and no FMA contraction:
 *     gcc -O3 -msse4 -mavx -ffp-contract=off -fopenmp -fPIC -shared      (CMakeLists.txt:4)
 * so that element-wise fp32 results are bit-identical to the reference's SSE/AVX code.
 */
#include "ictrack_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define LIEALG_SIGTHRESH 1e-4   /* utilities.h:22 */
#define LIEALG_EPSILON 1e-10    /* utilities.h:23 */
#define SSEMULTIPL 4            /* utilities.h:16 */

/* ------------------------------------------------------------------------------------------------
 * Reductions standing in for Eigen's DenseBase::sum() on a contiguous float vector.
 * Eigen is NOT in /root/reference (unpinned include dir, CMakeLists.txt:8,11-12).  This follows the
 * published algorithm of Eigen 3.3 Core/Redux.h, redux_impl<Func,Derived,LinearVectorizedTraversal,
 * NoUnrolling>::run — two packet accumulators over the aligned body, packet_res0+packet_res1, one odd
 * packet, predux, scalar tail — with predux<Packet4f> = (a0+a2)+(a1+a3) (SSE/PacketMath.h) and
 * predux<Packet8f> = predux4(lo+hi) (AVX/PacketMath.h).  Call sites: odometer.cpp:399-404, 430-455,
 * utilities.cpp:112,188.
 * ------------------------------------------------------------------------------------------------ */
static int g_sum_mode = 0;
void ict_oracle_set_sum_mode(int mode) { g_sum_mode = mode; }
int ict_oracle_get_sum_mode(void) { return g_sum_mode; }

#define DEF_PACKET_SUM(NAME, W, ELEM)                                                             \
  static float NAME(const float* a, const float* b, int64_t n) {                                  \
    (void)b;                                                                                      \
    const int64_t as2 = (n / (2 * W)) * (2 * W), as1 = (n / W) * W;                               \
    float res;                                                                                    \
    if (n == 0) return 0.0f;                                                                      \
    if (as1) {                                                                                    \
      float p0[W], p1[W];                                                                         \
      for (int k = 0; k < W; ++k) { const int64_t i = k; p0[k] = ELEM; }                          \
      if (as1 > W) {                                                                              \
        for (int k = 0; k < W; ++k) { const int64_t i = W + k; p1[k] = ELEM; }                    \
        for (int64_t idx = 2 * W; idx < as2; idx += 2 * W) {                                      \
          for (int k = 0; k < W; ++k) { const int64_t i = idx + k; p0[k] = p0[k] + ELEM; }        \
          for (int k = 0; k < W; ++k) { const int64_t i = idx + W + k; p1[k] = p1[k] + ELEM; }    \
        }                                                                                         \
        for (int k = 0; k < W; ++k) p0[k] = p0[k] + p1[k];                                        \
        if (as1 > as2)                                                                            \
          for (int k = 0; k < W; ++k) { const int64_t i = as2 + k; p0[k] = p0[k] + ELEM; }        \
      }                                                                                           \
      if (W == 8)                                                                                 \
        for (int k = 0; k < 4; ++k) p0[k] = p0[k] + p0[k + 4];                                    \
      res = (p0[0] + p0[2]) + (p0[1] + p0[3]);                                                    \
      for (int64_t i = as1; i < n; ++i) res = res + ELEM;                                         \
    } else {                                                                                      \
      { const int64_t i = 0; res = ELEM; }                                                        \
      for (int64_t i = 1; i < n; ++i) res = res + ELEM;                                           \
    }                                                                                             \
    return res;                                                                                   \
  }

DEF_PACKET_SUM(sum_p4, 4, a[i])
DEF_PACKET_SUM(sum_p8, 8, a[i])
DEF_PACKET_SUM(prodsum_p4, 4, (a[i] * b[i]))
DEF_PACKET_SUM(prodsum_p8, 8, (a[i] * b[i]))

static float esum(const float* a, int64_t n) {
  switch (g_sum_mode) {
    case 1: return sum_p8(a, 0, n);
    case 2: { double s = 0; for (int64_t i = 0; i < n; ++i) s += (double)a[i]; return (float)s; }
    case 3: { float s = 0; for (int64_t i = 0; i < n; ++i) s = s + a[i]; return s; }
    default: return sum_p4(a, 0, n);
  }
}
/* (x.array() * y.array()).sum(): the product is rounded to fp32 per element before it is added */
static float eprodsum(const float* a, const float* b, int64_t n) {
  switch (g_sum_mode) {
    case 1: return prodsum_p8(a, b, n);
    case 2: { double s = 0; for (int64_t i = 0; i < n; ++i) { float p = a[i] * b[i]; s += (double)p; } return (float)s; }
    case 3: { float s = 0; for (int64_t i = 0; i < n; ++i) { float p = a[i] * b[i]; s = s + p; } return s; }
    default: return prodsum_p4(a, b, n);
  }
}
float ict_oracle_sum(const float* a, int64_t n) { return esum(a, n); }

/* ------------------------------------------------------------------------------------------------
 * util_SE3_coeff_to_group<T>, utilities.h:84-145.  T=float: the unqualified sqrt/sin/cos/acos/tan calls
 * in the templates bind to the double C functions (fundamental types get no ADL and only ::sin(double) is
 * visible where the template is defined when the headers above it pull in <cmath>, as Eigen/Core does), so
 * the transcendental AND the expression around it (sin(sig)/sig ...) are evaluated in double and narrowed on
 * assignment.  That is what g++ 13 does with the reference sources in this container; verified
 * bit-identical against oracle/_ref in tests/test_oracle_vs_ref.py.
 * ------------------------------------------------------------------------------------------------ */
#define DEF_SE3_EXP(NAME, T)                                                                           \
  void NAME(T* cpos_G, const T* cpos_p) {                                                              \
    T ra1 = cpos_p[3] * cpos_p[3];                                                                     \
    T ra2 = cpos_p[4] * cpos_p[4];                                                                     \
    T ra3 = cpos_p[5] * cpos_p[5];                                                                     \
    T sig = (T)sqrt((double)(T)(ra1 + ra2 + ra3));                                                     \
    T sa, sb, sc;                                                                                      \
    T sigsq2 = (sig * sig);                                                                            \
    T sigsq3 = (sig * sig * sig);                                                                      \
    if (sig > LIEALG_SIGTHRESH) {                                                                      \
      sa = (T)(sin((double)sig) / (double)sig);                                                        \
      sb = (T)((1 - cos((double)sig)) / (double)sigsq2);                                               \
      sc = (T)(((double)sig - sin((double)sig)) / (double)sigsq3);                                     \
    } else {                                                                                           \
      sa = 1 - sigsq2 / 6 * (1 - sigsq2 / 20 * (1 - sigsq2 / 42));                                     \
      sb = (T)(.5 * (1 - sigsq2 / 12 * (1 - sigsq2 / 30 * (1 - sigsq2 / 56))));                        \
      sc = (1 - sigsq2 / 20 * (1 - sigsq2 / 42 * (1 - sigsq2 / 72))) / 6;                              \
    }                                                                                                  \
    T tmp1 = ra2 * sb;                                                                                 \
    T tmp2 = ra3 * sb;                                                                                 \
    T tmp3 = ra1 * sb;                                                                                 \
    T tmp4 = cpos_p[3] * cpos_p[4] * sb;                                                               \
    T tmp5 = cpos_p[5] * sa;                                                                           \
    T tmp6 = cpos_p[3] * cpos_p[5] * sb;                                                               \
    T tmp7 = cpos_p[4] * sa;                                                                           \
    T tmp8 = cpos_p[3] * sa;                                                                           \
    T tmp9 = cpos_p[4] * cpos_p[5] * sb;                                                               \
    cpos_G[0] = 1 - tmp1 - tmp2;                                                                       \
    cpos_G[1] = tmp4 - tmp5;                                                                           \
    cpos_G[2] = tmp7 + tmp6;                                                                           \
    cpos_G[4] = tmp5 + tmp4;                                                                           \
    cpos_G[5] = 1 - tmp3 - tmp2;                                                                       \
    cpos_G[6] = tmp9 - tmp8;                                                                           \
    cpos_G[8] = tmp6 - tmp7;                                                                           \
    cpos_G[9] = tmp8 + tmp9;                                                                           \
    cpos_G[10] = 1 - tmp3 - tmp1;                                                                      \
    tmp1 = cpos_p[5] * sb;                                                                             \
    tmp2 = cpos_p[3] * cpos_p[4] * sc;                                                                 \
    tmp3 = cpos_p[4] * sb;                                                                             \
    tmp4 = cpos_p[3] * cpos_p[5] * sc;                                                                 \
    tmp5 = cpos_p[3] * sb;                                                                             \
    tmp6 = cpos_p[4] * cpos_p[5] * sc;                                                                 \
    cpos_G[3] = (1 - (ra2 + ra3) * sc) * cpos_p[0] + (tmp2 - tmp1) * cpos_p[1] + (tmp3 + tmp4) * cpos_p[2]; \
    cpos_G[7] = (tmp1 + tmp2) * cpos_p[0] + (1 - (ra1 + ra3) * sc) * cpos_p[1] + (tmp6 - tmp5) * cpos_p[2]; \
    cpos_G[11] = (tmp4 - tmp3) * cpos_p[0] + (tmp5 + tmp6) * cpos_p[1] + (1 - (ra1 + ra2) * sc) * cpos_p[2]; \
  }
DEF_SE3_EXP(ict_oracle_se3_exp_f, float)
DEF_SE3_EXP(ict_oracle_se3_exp_d, double)

/* util_SE3_group_to_coeff<T>, utilities.h:149-241 */
#define DEF_SE3_LOG(NAME, T)                                                                           \
  void NAME(T* cpos_p, const T* cpos_G) {                                                              \
    T trace = cpos_G[0] + cpos_G[5] + cpos_G[10];                                                      \
    T theta = (T)acos((double)(T)(0.5f * (trace - 1)));                                                \
    T omega_hat[9], omega_hat_sq[9], V_inv[9];                                                         \
    memset(omega_hat, 0, sizeof(T) * 9);                                                               \
    if (theta < LIEALG_EPSILON) {                                                                      \
      cpos_p[3] = 0.0f;                                                                                \
      cpos_p[4] = 0.0f;                                                                                \
      cpos_p[5] = 0.0f;                                                                                \
      memset(omega_hat_sq, 0, sizeof(T) * 9);                                                          \
    } else {                                                                                           \
      T coef = (T)((double)theta / ((double)2.0f * sin((double)theta)));                               \
      omega_hat[1] = coef * (cpos_G[1] - cpos_G[4]);                                                   \
      omega_hat[3] = -omega_hat[1];                                                                    \
      omega_hat[2] = coef * (cpos_G[2] - cpos_G[8]);                                                   \
      omega_hat[6] = -omega_hat[2];                                                                    \
      omega_hat[5] = coef * (cpos_G[6] - cpos_G[9]);                                                   \
      omega_hat[7] = -omega_hat[5];                                                                    \
      cpos_p[3] = -omega_hat[5];                                                                       \
      cpos_p[4] = omega_hat[2];                                                                        \
      cpos_p[5] = -omega_hat[1];                                                                       \
      T omsq1 = omega_hat[1] * omega_hat[1];                                                           \
      T omsq2 = omega_hat[2] * omega_hat[2];                                                           \
      T omsq3 = omega_hat[5] * omega_hat[5];                                                           \
      omega_hat_sq[0] = -omsq1 - omsq2;                                                                \
      omega_hat_sq[1] = -omega_hat[2] * omega_hat[5];                                                  \
      omega_hat_sq[3] = omega_hat_sq[1];                                                               \
      omega_hat_sq[2] = omega_hat[1] * omega_hat[5];                                                   \
      omega_hat_sq[6] = omega_hat_sq[2];                                                               \
      omega_hat_sq[4] = -omsq1 - omsq3;                                                                \
      omega_hat_sq[5] = -omega_hat[1] * omega_hat[2];                                                  \
      omega_hat_sq[7] = omega_hat_sq[5];                                                               \
      omega_hat_sq[8] = -omsq2 - omsq3;                                                                \
    }                                                                                                  \
    T theta_help;                                                                                      \
    if (theta < LIEALG_SIGTHRESH)                                                                      \
      theta_help = 1.0f / 12.0f;                                                                       \
    else                                                                                               \
      theta_help = (T)(((double)1.0f - (double)theta / ((double)2.0f * tan((double)(T)(theta / 2.0f)))) / \
                       (double)(T)(theta * theta));                                                    \
    V_inv[0] = 1.0f + theta_help * omega_hat_sq[0];                                                    \
    V_inv[1] = -0.5f * omega_hat[1] + theta_help * omega_hat_sq[1];                                    \
    V_inv[2] = -0.5f * omega_hat[2] + theta_help * omega_hat_sq[2];                                    \
    V_inv[3] = -0.5f * omega_hat[3] + theta_help * omega_hat_sq[3];                                    \
    V_inv[4] = 1.0f + theta_help * omega_hat_sq[4];                                                    \
    V_inv[5] = -0.5f * omega_hat[5] + theta_help * omega_hat_sq[5];                                    \
    V_inv[6] = -0.5f * omega_hat[6] + theta_help * omega_hat_sq[6];                                    \
    V_inv[7] = -0.5f * omega_hat[7] + theta_help * omega_hat_sq[7];                                    \
    V_inv[8] = 1.0f + theta_help * omega_hat_sq[8];                                                    \
    cpos_p[0] = V_inv[0] * cpos_G[3] + V_inv[1] * cpos_G[7] + V_inv[2] * cpos_G[11];                   \
    cpos_p[1] = V_inv[3] * cpos_G[3] + V_inv[4] * cpos_G[7] + V_inv[5] * cpos_G[11];                   \
    cpos_p[2] = V_inv[6] * cpos_G[3] + V_inv[7] * cpos_G[7] + V_inv[8] * cpos_G[11];                   \
  }
DEF_SE3_LOG(ict_oracle_se3_log_f, float)
DEF_SE3_LOG(ict_oracle_se3_log_d, double)

/* ------------------------------------------------------------------------------------------------
 * CamClass::CamClass, camera.cpp:14-45.  out[8*l+..] = fx fy cx cy swo sho sw sh
 * ------------------------------------------------------------------------------------------------ */
void ict_oracle_camera_levels(int noscales, const float fc[2], const float cc[2], const int wh[2], int padding,
                              float* out) {
  for (int i = 0; i < noscales; ++i) {
    float sc_fct = (float)(1 / pow(2, i)); /* camera.cpp:34 */
    float* o = out + 8 * i;
    o[0] = sc_fct * fc[0];
    o[1] = sc_fct * fc[1];
    o[2] = sc_fct * cc[0];
    o[3] = sc_fct * cc[1];
    o[4] = sc_fct * (float)wh[0];
    o[5] = sc_fct * (float)wh[1];
    o[6] = o[4] + 2 * padding; /* camera.cpp:41 */
    o[7] = o[5] + 2 * padding;
  }
}

/* ------------------------------------------------------------------------------------------------
 * util_constructpyramide, utilities.cpp:14-52.  OpenCV is NOT in /root/reference; restated from the
 * documented behaviour of the three calls and pinned bit-exact against Python cv2 4.13 on uint8-valued
 * images (tests/golden/pyramid_*.npz):
 *   cv::resize(.5,.5,INTER_LINEAR) on an exact factor 2 takes OpenCV's area-fast path = 2x2 mean,
 *     ((a+b)+(c+d))*0.25 (utilities.cpp:24);
 *   cv::Sobel(ksize=1) = [-1 0 1], BORDER_DEFAULT=REFLECT_101 => 0 on the first/last column/row (:30-31);
 *   copyMakeBorder REPLICATE for the image (:40), CONSTANT 0 for the gradients (:45-46).
 * ------------------------------------------------------------------------------------------------ */
void ict_oracle_pyramid_build(const float* img, int w, int h, int lv_f, int pad,
                              float* out_I, float* out_dx, float* out_dy) {
  int64_t off[ICT_MAX_LEVELS];
  int sw[ICT_MAX_LEVELS], sh[ICT_MAX_LEVELS];
  int64_t tot = 0;
  for (int l = 0; l <= lv_f; ++l) {
    sw[l] = (w >> l) + 2 * pad;
    sh[l] = (h >> l) + 2 * pad;
    off[l] = tot;
    tot += (int64_t)sw[l] * sh[l];
  }
  float* prev = (float*)malloc(sizeof(float) * (size_t)w * h);
  float* cur = (float*)malloc(sizeof(float) * (size_t)w * h);
  memcpy(prev, img, sizeof(float) * (size_t)w * h);
  for (int l = 0; l <= lv_f; ++l) {
    const int lw = w >> l, lh = h >> l;
    if (l > 0) {
      const int pw = w >> (l - 1);
      for (int y = 0; y < lh; ++y)
        for (int x = 0; x < lw; ++x) {
          const float* r0 = prev + (size_t)(2 * y) * pw + 2 * x;
          const float* r1 = r0 + pw;
          cur[(size_t)y * lw + x] = ((r0[0] + r0[1]) + (r1[0] + r1[1])) * 0.25f;
        }
      float* t = prev; prev = cur; cur = t;
    }
    float* I = out_I + off[l];
    float* dx = out_dx ? out_dx + off[l] : 0;
    float* dy = out_dy ? out_dy + off[l] : 0;
    for (int Y = 0; Y < sh[l]; ++Y)
      for (int X = 0; X < sw[l]; ++X) {
        int y = Y - pad, x = X - pad;
        int yc = y < 0 ? 0 : (y >= lh ? lh - 1 : y);
        int xc = x < 0 ? 0 : (x >= lw ? lw - 1 : x);
        I[(size_t)Y * sw[l] + X] = prev[(size_t)yc * lw + xc];
        int inside = (x >= 0) & (x < lw) & (y >= 0) & (y < lh);
        if (dx) {
          float g = 0.0f;
          if (inside && x > 0 && x < lw - 1) g = prev[(size_t)y * lw + x + 1] - prev[(size_t)y * lw + x - 1];
          dx[(size_t)Y * sw[l] + X] = g;
        }
        if (dy) {
          float g = 0.0f;
          if (inside && y > 0 && y < lh - 1) g = prev[(size_t)(y + 1) * lw + x] - prev[(size_t)(y - 1) * lw + x];
          dy[(size_t)Y * sw[l] + X] = g;
        }
      }
  }
  free(prev);
  free(cur);
}

/* ------------------------------------------------------------------------------------------------
 * util_getPatch, utilities.cpp:55-113 ; util_getPatch_grad, utilities.cpp:115-189
 * ------------------------------------------------------------------------------------------------ */
void ict_oracle_getpatch(const float* img, const float* mid_in, float* tmp_in, const ict_optparam* op, int width) {
  float resid[2], we[4];
  int pos[4];
  pos[0] = (int)ceilf(mid_in[0] + .00001f); /* utilities.cpp:66 */
  pos[1] = (int)ceilf(mid_in[1] + .00001f);
  pos[2] = (int)floorf(mid_in[0]);
  pos[3] = (int)floorf(mid_in[1]);
  resid[0] = mid_in[0] - (float)pos[2];
  resid[1] = mid_in[1] - (float)pos[3];
  we[0] = resid[0] * resid[1];
  we[1] = (1 - resid[0]) * resid[1];
  we[2] = resid[0] * (1 - resid[1]);
  we[3] = (1 - resid[0]) * (1 - resid[1]);
  float* tmp_it = tmp_in;
  const float* img_e = img + pos[0] + op->pszd2;
  const int lbo = pos[1] + op->pszd2, ubo = pos[1] + op->pszd2m3;
  const int lbi = pos[0] + op->pszd2, ubi = pos[0] + op->pszd2m3;
  for (int r = lbo; r <= ubo; ++r) {
    const float* img_a = img_e + (int64_t)r * width;
    const float* img_c = img_e + (int64_t)(r - 1) * width;
    const float* img_b = img_a - 1;
    const float* img_d = img_c - 1;
    for (int c = lbi; c <= ubi; ++c, ++tmp_it, ++img_a, ++img_b, ++img_c, ++img_d)
      (*tmp_it) = we[0] * (*img_a) + we[1] * (*img_b) + we[2] * (*img_c) + we[3] * (*img_d);
  }
  if (op->dopatchnorm) { /* utilities.cpp:111-112 */
    const float m = esum(tmp_in, op->novals) / op->novals;
    for (int k = 0; k < op->novals; ++k) tmp_in[k] -= m;
  }
}

void ict_oracle_getpatch_grad(const float* img, const float* img_dx, const float* img_dy, const float* mid_in,
                              float* t, float* tdx, float* tdy, const ict_optparam* op, int width) {
  float resid[2], we[4];
  int pos[4];
  pos[0] = (int)ceilf(mid_in[0] + .00001f); /* utilities.cpp:128 */
  pos[1] = (int)ceilf(mid_in[1] + .00001f);
  pos[2] = (int)floorf(mid_in[0]);
  pos[3] = (int)floorf(mid_in[1]);
  resid[0] = mid_in[0] - (float)pos[2];
  resid[1] = mid_in[1] - (float)pos[3];
  we[0] = resid[0] * resid[1];
  we[1] = (1 - resid[0]) * resid[1];
  we[2] = resid[0] * (1 - resid[1]);
  we[3] = (1 - resid[0]) * (1 - resid[1]);
  const int pos0tt = pos[0] + op->pszd2;
  const int lbo = pos[1] + op->pszd2, ubo = pos[1] + op->pszd2m3;
  const int lbi = pos0tt, ubi = pos[0] + op->pszd2m3;
  float* t0 = t;
  for (int r = lbo; r <= ubo; ++r) {
    const int64_t o1 = (int64_t)r * width + pos0tt, o2 = (int64_t)(r - 1) * width + pos0tt;
    const float *a = img + o1, *c = img + o2, *b = a - 1, *d = c - 1;
    const float *ax = img_dx + o1, *cx = img_dx + o2, *bx = ax - 1, *dx = cx - 1;
    const float *ay = img_dy + o1, *cy = img_dy + o2, *by = ay - 1, *dy = cy - 1;
    for (int col = lbi; col <= ubi; ++col, ++t, ++a, ++b, ++c, ++d, ++tdx, ++ax, ++bx, ++cx, ++dx, ++tdy, ++ay,
             ++by, ++cy, ++dy) {
      (*t) = we[0] * (*a) + we[1] * (*b) + we[2] * (*c) + we[3] * (*d);
      (*tdx) = we[0] * (*ax) + we[1] * (*bx) + we[2] * (*cx) + we[3] * (*dx);
      (*tdy) = we[0] * (*ay) + we[1] * (*by) + we[2] * (*cy) + we[3] * (*dy);
    }
  }
  if (op->dopatchnorm) { /* utilities.cpp:187-188: intensity only */
    const float m = esum(t0, op->novals) / op->novals;
    for (int k = 0; k < op->novals; ++k) t0[k] -= m;
  }
}

/* ------------------------------------------------------------------------------------------------
 * delta_p = Hes.fullPivLu().solve(sumsd), odometer.cpp:509-515.  Eigen is absent; this follows the
 * published algorithm of Eigen 3.3 LU/FullPivLU.h: computeInPlace() (column-major max search with strict
 * '>', row+column swaps, column scaling by the pivot, rank-1 update of the trailing block) and
 * _solve_impl() (rank from |pivot| > eps*6*|maxpivot|, unit-lower forward substitution, upper backward
 * substitution on the leading rank x rank block, both column-oriented, then the column permutation).
 * H is 6x6 column-major as in Eigen::Matrix<float,6,6>.
 * ------------------------------------------------------------------------------------------------ */
void ict_oracle_solve6(const float* H, const float* b, float* x) {
  float lu[36];
  int rowtr[6], coltr[6];
  memcpy(lu, H, sizeof(lu));
#define LU(i, j) lu[(i) + 6 * (j)]
  int nonzero_pivots = 6;
  float maxpivot = 0.0f;
  for (int k = 0; k < 6; ++k) {
    int pr = k, pc = k;
    float biggest = -1.0f;
    for (int j = k; j < 6; ++j)
      for (int i = k; i < 6; ++i) {
        float v = fabsf(LU(i, j));
        if (v > biggest) { biggest = v; pr = i; pc = j; }
      }
    if (biggest == 0.0f) {
      nonzero_pivots = k;
      for (int i = k; i < 6; ++i) { rowtr[i] = i; coltr[i] = i; }
      break;
    }
    if (biggest > maxpivot) maxpivot = biggest;
    rowtr[k] = pr;
    coltr[k] = pc;
    if (k != pr) for (int j = 0; j < 6; ++j) { float t = LU(k, j); LU(k, j) = LU(pr, j); LU(pr, j) = t; }
    if (k != pc) for (int i = 0; i < 6; ++i) { float t = LU(i, k); LU(i, k) = LU(i, pc); LU(i, pc) = t; }
    if (k < 5) {
      for (int i = k + 1; i < 6; ++i) LU(i, k) = LU(i, k) / LU(k, k);
      for (int j = k + 1; j < 6; ++j)
        for (int i = k + 1; i < 6; ++i) LU(i, j) = LU(i, j) - LU(i, k) * LU(k, j);
    }
  }
  /* permutations: P = T(0)..T(5) applied in order; Q accumulated the same way for columns */
  int rank = 0;
  {
    const float premult = fabsf(maxpivot) * (1.1920929e-07f * 6.0f);
    for (int i = 0; i < nonzero_pivots; ++i) rank += (fabsf(LU(i, i)) > premult);
  }
  if (rank == 0) { for (int i = 0; i < 6; ++i) x[i] = 0.0f; return; } /* _solve_impl uses rank() */
  float c[6];
  for (int i = 0; i < 6; ++i) c[i] = b[i];
  for (int k = 0; k < 6; ++k) if (rowtr[k] != k) { float t = c[k]; c[k] = c[rowtr[k]]; c[rowtr[k]] = t; }
  /* unit lower, column-oriented forward substitution */
  for (int i = 0; i < 6; ++i)
    for (int r = i + 1; r < 6; ++r) c[r] = c[r] - c[i] * LU(r, i);
  /* upper, leading rank x rank block, column-oriented backward substitution */
  for (int i = rank - 1; i >= 0; --i) {
    c[i] = c[i] / LU(i, i);
    for (int r = 0; r < i; ++r) c[r] = c[r] - c[i] * LU(r, i);
  }
  /* dst = Q*c, Q = T'_0 T'_1 ... T'_5 (column transpositions in elimination order), rows beyond the nonzero
   * pivots zeroed: apply the transpositions to c last-to-first */
  for (int i = rank; i < 6; ++i) c[i] = 0.0f;
  for (int k = 5; k >= 0; --k) if (coltr[k] != k) { float t = c[k]; c[k] = c[coltr[k]]; c[coltr[k]] = t; }
  for (int i = 0; i < 6; ++i) x[i] = c[i];
#undef LU
}

/* ------------------------------------------------------------------------------------------------
 * The odometer: CamClass (camera.h/.cpp) + PoseClass (pose.h/.cpp) + OdometerClass (odometer.h/.cpp)
 * ------------------------------------------------------------------------------------------------ */
struct ict_oracle_odom {
  const ict_optparam* op; /* borrowed, like the reference (pose.h:60, odometer.h:112) */
  int alloc_M, alloc_n, alloc_lvf;
  float cam[8 * ICT_MAX_LEVELS];
  /* PoseClass state, pose.h:51-55 */
  double p_meanshift[3], p_varval;
  float cpos_G[12], cpos_p[6];
  /* OdometerClass state, odometer.h:40-60 */
  double meanshift[3], varval;
  const float **img_ref, **img_ref_dx, **img_ref_dy, **img_new;
  int nopoints;
  float Hes[36], sumsd[6], delta_p[6];
  unsigned char *ind_ref, *ind_new;
  float *pt3d, *pt3d_ref, *pt2d[ICT_MAX_LEVELS], *pt2d_new;
  float *pat_ref, *pat_dx, *pat_dy, *pat_new, *sd[6], *sdp[6], *pdiff;
  /* instrumentation (not in the reference) */
  float* trace;
  int trace_cap, trace_n;
  int iters[ICT_MAX_LEVELS];
  int64_t npixres;
};

#define CAM_FX(o, l) ((o)->cam[8 * (l) + 0])
#define CAM_FY(o, l) ((o)->cam[8 * (l) + 1])
#define CAM_CX(o, l) ((o)->cam[8 * (l) + 2])
#define CAM_CY(o, l) ((o)->cam[8 * (l) + 3])
#define CAM_SWO(o, l) ((o)->cam[8 * (l) + 4])
#define CAM_SHO(o, l) ((o)->cam[8 * (l) + 5])
#define CAM_SW(o, l) ((o)->cam[8 * (l) + 6])

static float* alloc_f(size_t n) {
  void* p = 0;
  if (n == 0) n = 1;
  if (posix_memalign(&p, 64, sizeof(float) * n)) return 0;
  memset(p, 0, sizeof(float) * n);
  return (float*)p;
}

/* OdometerClass::ResetOdometer, odometer.cpp:580-609 */
static void reset_odometer(ict_oracle_odom* o) {
  const size_t mn = (size_t)o->alloc_M * o->alloc_n;
  memset(o->Hes, 0, sizeof(o->Hes));
  memset(o->ind_ref, 1, o->alloc_M);
  memset(o->ind_new, 1, o->alloc_M);
  memset(o->pat_ref, 0, sizeof(float) * mn);
  memset(o->pat_dx, 0, sizeof(float) * mn);
  memset(o->pat_dy, 0, sizeof(float) * mn);
  memset(o->pat_new, 0, sizeof(float) * mn);
  for (int k = 0; k < 6; ++k) {
    memset(o->sd[k], 0, sizeof(float) * mn);
    memset(o->sdp[k], 0, sizeof(float) * mn);
  }
}

/* OdometerClass::OdometerClass, odometer.cpp:19-154 (+ CamClass with padding = psz as both drivers do) */
ict_oracle_odom* ict_oracle_odom_create(const ict_optparam* op, const float fc[2], const float cc[2],
                                        const int wh[2]) {
  ict_oracle_odom* o = (ict_oracle_odom*)calloc(1, sizeof(*o));
  o->op = op;
  o->alloc_M = op->maxpttrack;
  o->alloc_n = op->novals;
  o->alloc_lvf = op->lv_f;
  ict_oracle_camera_levels(op->lv_f + 1, fc, cc, wh, op->psz, o->cam);
  const size_t M = (size_t)op->maxpttrack, mn = M * op->novals;
  o->pt3d = alloc_f(3 * M + 8);
  o->pt3d_ref = alloc_f(3 * M + 8);
  o->pt2d_new = alloc_f(2 * M + 8);
  for (int i = 0; i <= op->lv_f; ++i) o->pt2d[i] = alloc_f(2 * M + 8);
  o->pat_ref = alloc_f(mn);
  o->pat_dx = alloc_f(mn);
  o->pat_dy = alloc_f(mn);
  o->pat_new = alloc_f(mn);
  o->pdiff = alloc_f(op->novals);
  for (int k = 0; k < 6; ++k) { o->sd[k] = alloc_f(mn); o->sdp[k] = alloc_f(mn); }
  o->ind_ref = (unsigned char*)malloc(M + 1);
  o->ind_new = (unsigned char*)malloc(M + 1);
  reset_odometer(o);
  return o;
}

void ict_oracle_odom_destroy(ict_oracle_odom* o) {
  if (!o) return;
  free(o->pt3d); free(o->pt3d_ref); free(o->pt2d_new);
  for (int i = 0; i <= o->alloc_lvf; ++i) free(o->pt2d[i]);
  free(o->pat_ref); free(o->pat_dx); free(o->pat_dy); free(o->pat_new); free(o->pdiff);
  for (int k = 0; k < 6; ++k) { free(o->sd[k]); free(o->sdp[k]); }
  free(o->ind_ref); free(o->ind_new);
  free(o);
}

void ict_oracle_odom_set_trace(ict_oracle_odom* o, float* trace, int trace_cap) {
  o->trace = trace;
  o->trace_cap = trace_cap;
  o->trace_n = 0;
}

/* OdometerClass::Set3Dpoints, odometer.cpp:171-239 (mutates pt_in when donorm, :207-212) */
void ict_oracle_set3dpoints(ict_oracle_odom* o, double* pt_in, int nopoints_in) {
  const ict_optparam* op = o->op;
  reset_odometer(o);
  memset(o->meanshift, 0, sizeof(o->meanshift));
  o->varval = 0;
  float* q1 = o->pt3d;
  float* q2 = o->pt3d + op->maxpttrack;
  float* q3 = o->pt3d + 2 * op->maxpttrack;
  o->nopoints = nopoints_in < op->maxpttrack ? nopoints_in : op->maxpttrack;
  const int n = o->nopoints;
  double *p1 = pt_in, *p2 = pt_in + nopoints_in, *p3 = pt_in + 2 * (size_t)nopoints_in;
  if (op->donorm) {
    const double nd = (double)n;
    for (int i = 0; i < n; ++i) o->meanshift[0] += p1[i];
    for (int i = 0; i < n; ++i) o->meanshift[1] += p2[i];
    for (int i = 0; i < n; ++i) o->meanshift[2] += p3[i];
    o->meanshift[0] /= nd;
    o->meanshift[1] /= nd;
    o->meanshift[2] /= nd;
    for (int i = 0; i < n; ++i) {
      p1[i] -= o->meanshift[0];
      p2[i] -= o->meanshift[1];
      p3[i] -= o->meanshift[2];
      o->varval += p1[i] * p1[i] + p2[i] * p2[i] + p3[i] * p3[i];
    }
    o->varval /= nd;
    for (int i = 0; i < n; ++i) {
      q1[i] = (float)(p1[i] / o->varval);
      q2[i] = (float)(p2[i] / o->varval);
      q3[i] = (float)(p3[i] / o->varval);
    }
  } else {
    for (int i = 0; i < n; ++i) {
      q1[i] = (float)p1[i];
      q2[i] = (float)p2[i];
      q3[i] = (float)p3[i];
    }
  }
}

/* PoseClass::setpose_se3, pose.cpp:25-76 */
static void setpose_se3(ict_oracle_odom* o, const double* p_in, const double* meanshift_in, double varval_in) {
  double p[6];
  memcpy(p, p_in, sizeof(p));
  if (o->op->donorm) {
    o->p_varval = varval_in;
    memcpy(o->p_meanshift, meanshift_in, sizeof(double) * 3);
    double G[12], t[3];
    ict_oracle_se3_exp_d(G, p);
    t[0] = -G[0] * G[3] - G[4] * G[7] - G[8] * G[11];
    t[1] = -G[1] * G[3] - G[5] * G[7] - G[9] * G[11];
    t[2] = -G[2] * G[3] - G[6] * G[7] - G[10] * G[11];
    t[0] = (t[0] - o->p_meanshift[0]) / o->p_varval;
    t[1] = (t[1] - o->p_meanshift[1]) / o->p_varval;
    t[2] = (t[2] - o->p_meanshift[2]) / o->p_varval;
    G[3] = -G[0] * t[0] - G[1] * t[1] - G[2] * t[2];
    G[7] = -G[4] * t[0] - G[5] * t[1] - G[6] * t[2];
    G[11] = -G[8] * t[0] - G[9] * t[1] - G[10] * t[2];
    ict_oracle_se3_log_d(p, G);
  }
  for (int k = 0; k < 6; ++k) o->cpos_p[k] = (float)p[k];
  ict_oracle_se3_exp_f(o->cpos_G, o->cpos_p);
}

/* PoseClass::getPose_se3, pose.cpp:79-113 */
static void getpose_se3(const ict_oracle_odom* o, double* p_out) {
  float pu[6];
  memcpy(pu, o->cpos_p, sizeof(pu));
  if (o->op->donorm) {
    float G[12];
    memcpy(G, o->cpos_G, sizeof(G)); /* pose.cpp:88 copies sizeof(double)*6 == 12 floats */
    double t[3];
    t[0] = -G[0] * G[3] - G[4] * G[7] - G[8] * G[11]; /* fp32 expression, widened on assignment */
    t[1] = -G[1] * G[3] - G[5] * G[7] - G[9] * G[11];
    t[2] = -G[2] * G[3] - G[6] * G[7] - G[10] * G[11];
    t[0] = t[0] * o->p_varval + o->p_meanshift[0];
    t[1] = t[1] * o->p_varval + o->p_meanshift[1];
    t[2] = t[2] * o->p_varval + o->p_meanshift[2];
    G[3] = (float)(-G[0] * t[0] - G[1] * t[1] - G[2] * t[2]); /* float*double -> double, narrowed */
    G[7] = (float)(-G[4] * t[0] - G[5] * t[1] - G[6] * t[2]);
    G[11] = (float)(-G[8] * t[0] - G[9] * t[1] - G[10] * t[2]);
    ict_oracle_se3_log_f(pu, G);
  }
  for (int k = 0; k < 6; ++k) p_out[k] = (double)pu[k];
}

/* PoseClass::project_pt / project_pt_save_rotated, pose.cpp:307-397 / 400-488 (count rounded up to x4) */
static void project_pt(const ict_oracle_odom* o, const float* pt3d, float* pt3d_rot, float* pt2d, int nopoints,
                       int sc) {
  const int M = o->op->maxpttrack;
  const float fx = CAM_FX(o, sc), fy = CAM_FY(o, sc), cx = CAM_CX(o, sc), cy = CAM_CY(o, sc);
  const float* G = o->cpos_G;
  const int div = nopoints % SSEMULTIPL;
  if (div > 0) nopoints = nopoints + (SSEMULTIPL - div);
  const float *X = pt3d, *Y = pt3d + M, *Z = pt3d + 2 * M;
  float *x = pt2d, *y = pt2d + M;
  for (int i = 0; i < nopoints; ++i) {
    const float tx = G[0] * X[i] + G[1] * Y[i] + G[2] * Z[i] + G[3];
    const float ty = G[4] * X[i] + G[5] * Y[i] + G[6] * Z[i] + G[7];
    const float tz = G[8] * X[i] + G[9] * Y[i] + G[10] * Z[i] + G[11];
    if (pt3d_rot) {
      pt3d_rot[i] = tx;
      pt3d_rot[i + M] = ty;
      pt3d_rot[i + 2 * M] = tz;
    }
    x[i] = (tx / tz) * fx + cx;
    y[i] = (ty / tz) * fy + cy;
  }
}

/* OdometerClass::SetPose, odometer.cpp:241-255 */
void ict_oracle_setpose(ict_oracle_odom* o, const double* p_in, const float** img_ref, const float** img_ref_dx,
                        const float** img_ref_dy, const float** img_new) {
  const ict_optparam* op = o->op;
  o->img_ref = img_ref;
  o->img_ref_dx = img_ref_dx;
  o->img_ref_dy = img_ref_dy;
  o->img_new = img_new;
  setpose_se3(o, p_in, o->meanshift, o->varval);
  project_pt(o, o->pt3d, o->pt3d_ref, o->pt2d[op->lv_f], o->nopoints, op->lv_f);
  for (int sl = op->lv_f - 1; sl >= op->lv_l; --sl) project_pt(o, o->pt3d, 0, o->pt2d[sl], o->nopoints, sl);
}

/* OdometerClass::ComputeHessian, odometer.cpp:428-472 */
static void compute_hessian(ict_oracle_odom* o) {
  const int64_t mn = (int64_t)o->op->novals * o->op->maxpttrack;
  for (int a = 0; a < 6; ++a)
    for (int b = a; b < 6; ++b) {
      const float v = eprodsum(o->sd[a], o->sd[b], mn);
      o->Hes[a + 6 * b] = v;
      o->Hes[b + 6 * a] = v;
    }
}

/* OdometerClass::TrackPose, odometer.cpp:257-426 */
void ict_oracle_trackpose(ict_oracle_odom* o, double* p_out) {
  const ict_optparam* op = o->op;
  const int M = op->maxpttrack, n = op->novals, np = o->nopoints;
  const int64_t mn = (int64_t)M * n;
  o->npixres = 0;
  o->trace_n = 0;
  for (int sl = op->lv_f; sl >= op->lv_l; --sl) {
    const float swo = CAM_SWO(o, sl), sho = CAM_SHO(o, sl);
    const int width = (int)CAM_SW(o, sl); /* float getsw() passed as const int width, odometer.cpp:286 */
    /* 4. reference patches + gradients, odometer.cpp:268-298 */
    for (int i = 0; i < np; ++i) {
      float mid[2] = {o->pt2d[sl][i], o->pt2d[sl][i + M]};
      /* The reference tests (x < 0) | (y < 0) | (x > swo) | (y > sho): the same for finite x, y, but a NaN placement
       * (donorm on one point or on equal points, include/ictrack.h) would pass it and be sampled.  Negated, as in the
       * kernels, NaN is outside. */
      if (!((mid[0] >= 0) & (mid[1] >= 0) & (mid[0] <= swo) & (mid[1] <= sho))) {
        o->ind_ref[i] = 0;
      } else {
        o->ind_ref[i] = 1;
        ict_oracle_getpatch_grad(o->img_ref[sl], o->img_ref_dx[sl], o->img_ref_dy[sl], mid,
                                 o->pat_ref + (size_t)i * n, o->pat_dx + (size_t)i * n,
                                 o->pat_dy + (size_t)i * n, op, width);
      }
    }
    /* 5. steepest-descent images, odometer.cpp:302-328 */
    for (int i = 0; i < np; ++i) {
      if (!o->ind_ref[i]) continue;
      const float pt_x = o->pt3d_ref[i], pt_y = o->pt3d_ref[i + M], pt_z = o->pt3d_ref[i + 2 * M];
      const float pt_zsq = pt_z * pt_z;
      const float fx = CAM_FX(o, sl), fy = CAM_FY(o, sl);
      const float c1x = (fx / pt_z);
      const float c2y = (fy / pt_z);
      const float c3x = (-pt_x / pt_zsq * fx), c3y = (-pt_y / pt_zsq * fy);
      const float c4x = (-pt_x * pt_y / pt_zsq * fx);
      const float c4y = (float)((-(1.0 + pt_y * pt_y / pt_zsq)) * fy); /* double, narrowed by Eigen's scalar op */
      const float c5x = (float)((1.0 + pt_x * pt_x / pt_zsq) * fx);
      const float c5y = (pt_x * pt_y / pt_zsq * fy);
      const float c6x = (-pt_y / pt_z * fx), c6y = (pt_x / pt_z * fy);
      const float* dx = o->pat_dx + (size_t)i * n;
      const float* dy = o->pat_dy + (size_t)i * n;
      float* s1 = o->sd[0] + (size_t)i * n; float* s2 = o->sd[1] + (size_t)i * n;
      float* s3 = o->sd[2] + (size_t)i * n; float* s4 = o->sd[3] + (size_t)i * n;
      float* s5 = o->sd[4] + (size_t)i * n; float* s6 = o->sd[5] + (size_t)i * n;
      for (int k = 0; k < n; ++k) {
        s1[k] = dx[k] * c1x;
        s2[k] = dy[k] * c2y;
        s3[k] = dx[k] * c3x + dy[k] * c3y;
        s4[k] = dx[k] * c4x + dy[k] * c4y;
        s5[k] = dx[k] * c5x + dy[k] * c5y;
        s6[k] = dx[k] * c6x + dy[k] * c6y;
      }
    }
    /* 6. Hessian */
    compute_hessian(o);

    float normdp_init = 1e-10; /* odometer.cpp:341-342 */
    float normdp = normdp_init;
    int it;
    for (it = 0; (it < op->maxiter) & ((normdp / normdp_init) > op->normdp_ratio); ++it) {
      for (int k = 0; k < 6; ++k) memset(o->sdp[k], 0, sizeof(float) * mn); /* :352-357 */
      project_pt(o, o->pt3d, 0, o->pt2d_new, np, sl);                        /* :360 */
      int nvis = 0;
      double abssum[6] = {0, 0, 0, 0, 0, 0};
      for (int i = 0; i < np; ++i) { /* :363-396 */
        float mid[2] = {o->pt2d_new[i], o->pt2d_new[i + M]};
        if (!((mid[0] >= 0) & (mid[1] >= 0) & (mid[0] <= swo) & (mid[1] <= sho))) { /* NaN: outside (see 4.) */
          o->ind_new[i] = 0;
        } else {
          o->ind_new[i] = 1;
          ++nvis;
          float* pn = o->pat_new + (size_t)i * n;
          ict_oracle_getpatch(o->img_new[sl], mid, pn, op, width);
          const float* pr = o->pat_ref + (size_t)i * n;
          float* pd = o->pdiff;
          for (int k = 0; k < n; ++k) pd[k] = pr[k] - pn[k];
          for (int a = 0; a < 6; ++a) {
            const float* s = o->sd[a] + (size_t)i * n;
            float* sp = o->sdp[a] + (size_t)i * n;
            for (int k = 0; k < n; ++k) sp[k] = s[k] * pd[k];
            if (o->trace) { /* instrumentation only: sum |sd_k * pdiff|, the scale of the summation noise */
              double as = 0;
              for (int k = 0; k < n; ++k) as += fabs((double)sp[k]);
              abssum[a] += as;
            }
          }
        }
      }
      for (int a = 0; a < 6; ++a) o->sumsd[a] = esum(o->sdp[a], mn); /* 9a :399-404 */
      ict_oracle_solve6(o->Hes, o->sumsd, o->delta_p);               /* 9b :407 */
      for (int a = 0; a < 6; ++a) o->cpos_p[a] += o->delta_p[a];     /* 10 addpose_se3, pose.cpp:116-129 */
      ict_oracle_se3_exp_f(o->cpos_G, o->cpos_p);
      { /* delta_p.lpNorm<1>(), :412 — Eigen 3.3 fixed-size redux: predux(first Packet4f) + pairwise remainder */
        const float* d = o->delta_p;
        normdp = ((fabsf(d[0]) + fabsf(d[2])) + (fabsf(d[1]) + fabsf(d[3]))) + (fabsf(d[4]) + fabsf(d[5]));
      }
      if (it == 0) normdp_init = normdp;
      o->npixres += (int64_t)nvis * n;
      if (o->trace && o->trace_n < o->trace_cap) {
        float* r = o->trace + (size_t)ICT_TRACE_FLOATS * o->trace_n++;
        r[0] = (float)sl;
        r[1] = (float)it;
        for (int a = 0; a < 6; ++a) { r[2 + a] = o->sumsd[a]; r[8 + a] = o->delta_p[a]; }
        r[14] = normdp;
        r[15] = (float)nvis;
        for (int a = 0; a < 6; ++a) r[16 + a] = (float)abssum[a];
        r[22] = r[23] = 0.0f;
      }
    }
    o->iters[op->lv_f - sl] = it;
  }
  if (o->trace)
    for (int k = o->trace_n; k < o->trace_cap; ++k) {
      float* r = o->trace + (size_t)ICT_TRACE_FLOATS * k;
      memset(r, 0, sizeof(float) * ICT_TRACE_FLOATS);
      r[0] = -1.0f;
    }
  getpose_se3(o, p_out);
}

const float* ict_oracle_get2dpoints(const ict_oracle_odom* o) { return o->pt2d[o->op->lv_l]; }
const int* ict_oracle_last_iters(const ict_oracle_odom* o) { return o->iters; }
int64_t ict_oracle_last_npixres(const ict_oracle_odom* o) { return o->npixres; }
const float* ict_oracle_hessian(const ict_oracle_odom* o) { return o->Hes; }

/* ------------------------------------------------------------------------------------------------
 * Batch of independent tracks (the sid loop of run_track_nposes.cpp:193 generalised): one odometer per
 * OpenMP thread, tracks distributed dynamically.
 * ------------------------------------------------------------------------------------------------ */
int ict_oracle_track_batch(const ict_optparam* op, const float fc[2], const float cc[2], const int wh[2],
                           int nframes, const float* const* planes_I, const float* const* planes_dx,
                           const float* const* planes_dy, int T, const int64_t* pt_off, const double* pts,
                           const int* ref_frame, const int* new_frame, const double* p_in, double* p_out,
                           int* iters, float* trace, int trace_cap, int64_t* npixres, float* pt2d_out,
                           int nthreads) {
  int64_t off[ICT_MAX_LEVELS];
  int64_t tot = 0;
  const int L = op->lv_f - op->lv_l + 1;
  for (int l = 0; l <= op->lv_f; ++l) {
    off[l] = tot;
    tot += (int64_t)((wh[0] >> l) + 2 * op->psz) * ((wh[1] >> l) + 2 * op->psz);
  }
  (void)nframes;
#ifdef _OPENMP
  if (nthreads <= 0) nthreads = omp_get_max_threads();
#else
  nthreads = 1;
#endif
#pragma omp parallel num_threads(nthreads)
  {
    ict_oracle_odom* o = ict_oracle_odom_create(op, fc, cc, wh);
    int64_t maxn = 0;
    for (int t = 0; t < T; ++t) if (pt_off[t + 1] - pt_off[t] > maxn) maxn = pt_off[t + 1] - pt_off[t];
    double* buf = (double*)malloc(sizeof(double) * 3 * (size_t)(maxn ? maxn : 1));
    const float *ri[ICT_MAX_LEVELS], *rx[ICT_MAX_LEVELS], *ry[ICT_MAX_LEVELS], *ni[ICT_MAX_LEVELS];
#pragma omp for schedule(dynamic, 4)
    for (int t = 0; t < T; ++t) {
      const int n = (int)(pt_off[t + 1] - pt_off[t]);
      memcpy(buf, pts + 3 * pt_off[t], sizeof(double) * 3 * (size_t)n);
      for (int l = 0; l <= op->lv_f; ++l) {
        ri[l] = planes_I[ref_frame[t]] + off[l];
        rx[l] = planes_dx[ref_frame[t]] + off[l];
        ry[l] = planes_dy[ref_frame[t]] + off[l];
        ni[l] = planes_I[new_frame[t]] + off[l];
      }
      if (trace) ict_oracle_odom_set_trace(o, trace + (size_t)t * trace_cap * ICT_TRACE_FLOATS, trace_cap);
      ict_oracle_set3dpoints(o, buf, n);
      ict_oracle_setpose(o, p_in + 6 * (size_t)t, ri, rx, ry, ni);
      if (pt2d_out) {
        const float* q = ict_oracle_get2dpoints(o);
        const int nn = n < op->maxpttrack ? n : op->maxpttrack;
        for (int i = 0; i < nn; ++i) {
          pt2d_out[2 * pt_off[t] + i] = q[i];
          pt2d_out[2 * pt_off[t] + n + i] = q[i + op->maxpttrack];
        }
      }
      ict_oracle_trackpose(o, p_out + 6 * (size_t)t);
      if (iters) memcpy(iters + (size_t)t * L, o->iters, sizeof(int) * L);
      if (npixres) npixres[t] = o->npixres;
    }
    free(buf);
    ict_oracle_odom_destroy(o);
  }
  return 0;
}

/* ------------------------------------------------------------------------------------------------
 * NCC hypothesis scoring, run_track_nposes.cpp:271-355 (one pose sample).  Patches persist across
 * points exactly like patch_b/patch_r/patch_f there; "/= norm()" is Eigen 3.3's true division.
 * ------------------------------------------------------------------------------------------------ */
void ict_oracle_ncc_score(const ict_optparam* op_in, const float fc[2], const float cc[2], const int wh[2],
                          const float* img_b, const float* img_r, const float* img_f, int nback, int nfwd,
                          const float* pt2d_back, const float* pt2d_refe, const float* pt2d_forw, int n,
                          float* out_corr) {
  ict_optparam op = *op_in;
  op.dopatchnorm = 1; /* run_track_nposes.cpp:281 */
  float cam[8 * ICT_MAX_LEVELS];
  ict_oracle_camera_levels(op.lv_f + 1, fc, cc, wh, op.psz, cam);
  const float swo = cam[8 * op.lv_l + 4], sho = cam[8 * op.lv_l + 5];
  const int width = (int)cam[8 * op.lv_l + 6];
  const int nv = op.novals;
  float* pb = alloc_f(nv);
  float* pr = alloc_f(nv);
  float* pf = alloc_f(nv);
  for (int i = 0; i < n; ++i) {
    int b_val = 1, r_val = 1, f_val = 1;
    float mid[2], weight[2];
    mid[0] = pt2d_back[i]; mid[1] = pt2d_back[i + n];
    if ((mid[0] > 0) & (mid[1] > 0) & (mid[0] < swo) & (mid[1] < sho)) ict_oracle_getpatch(img_b, mid, pb, &op, width);
    else b_val = 0;
    mid[0] = pt2d_refe[i]; mid[1] = pt2d_refe[i + n];
    if ((mid[0] > 0) & (mid[1] > 0) & (mid[0] < swo) & (mid[1] < sho)) ict_oracle_getpatch(img_r, mid, pr, &op, width);
    else r_val = 0;
    mid[0] = pt2d_forw[i]; mid[1] = pt2d_forw[i + n];
    if ((mid[0] > 0) & (mid[1] > 0) & (mid[0] < swo) & (mid[1] < sho)) ict_oracle_getpatch(img_f, mid, pf, &op, width);
    else f_val = 0;
    float corr = -1;
    if (r_val) {
      const float nb = sqrtf(eprodsum(pb, pb, nv)), nr = sqrtf(eprodsum(pr, pr, nv)), nf = sqrtf(eprodsum(pf, pf, nv));
      for (int k = 0; k < nv; ++k) { pb[k] = pb[k] / nb; pr[k] = pr[k] / nr; pf[k] = pf[k] / nf; }
      float corr_br, corr_rf;
      if (b_val) { float s = eprodsum(pb, pr, nv); corr_br = 0.0f < s ? s : 0.0f; weight[0] = (float)(nback * nback); }
      else { corr_br = -1; weight[0] = 0; }
      if (f_val) { float s = eprodsum(pr, pf, nv); corr_rf = 0.0f < s ? s : 0.0f; weight[1] = (float)(nfwd * nfwd); }
      else { corr_rf = -1; weight[1] = 0; }
      const float v = (corr_br * weight[0] + corr_rf * weight[1]) / (weight[0] + weight[1]);
      corr = 0.0f < v ? v : 0.0f;
    }
    out_corr[i] = corr;
  }
  free(pb); free(pr); free(pf);
}
