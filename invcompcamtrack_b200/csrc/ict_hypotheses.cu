// ict_hypotheses.cu — pose hypotheses from minimal 4-point samples + their inlier sets: the step that FEEDS the N-pose
// tracker (SURVEY.md §8 f3; func_ransac_fitcameras_odom.m:29-90: sample 4 correspondences, reject degenerate samples,
// solve the pose, reproject all points, keep the inliers within inlthresh, reject samples with fewer than 4).
//
// The reference solves the minimal problem with the external ASPnP toolbox (absent from the reference tree, MATLAB,
// Groebner-basis solver): there is nothing to restate.  What is built here has the same role and interface with a
// solver that suits a batch on a GPU: every sample runs a damped Gauss-Newton on the reprojection error of its four
// points (8 equations, 6 unknowns) in fp64 from a common initial pose — in the tracker's use the pose of the reference
// frame, from which the hypotheses are a few pixels away — with the left-multiplied twist G <- exp(xi) G that
// util_SE3_coeff_to_group (utilities.h:84-145) parameterises.  One thread per sample for the solve, one CTA per sample
// for the reprojection of all correspondences.  oracle/hypotheses.py is the numpy statement of the same algorithm.
#include "ict_kernels.cuh"
#include "ict_device.cuh"

namespace ict {


struct HypArgs {
  double fx, fy, cx, cy;
  int npts, nsamples, maxiter;
  double inlthresh;
  const double* pt2d;      // [2][npts]: x block, y block
  const double* pt3d;      // [3][npts]
  const int* sample;       // [nsamples][4], 0-based
  double p_init[6];
  double* pose;            // [nsamples][6]
  int* status;             // [nsamples]: 1 solved, 0 degenerate sample / no convergence / point behind the camera
  int* ninl;               // [nsamples]
  unsigned char* mask;     // [nsamples][npts]
};

// solve A x = b for a symmetric positive definite 6x6 (A is overwritten); false when a pivot vanishes
__device__ bool hyp_solve6(double* A, double* b, double* x) {
  for (int k = 0; k < 6; ++k) {
    int piv = k;
    double best = fabs(A[k * 6 + k]);
    for (int i = k + 1; i < 6; ++i)
      if (fabs(A[i * 6 + k]) > best) { best = fabs(A[i * 6 + k]); piv = i; }
    if (!(best > 1e-300)) return false;
    if (piv != k) {
      for (int j = 0; j < 6; ++j) { const double t = A[k * 6 + j]; A[k * 6 + j] = A[piv * 6 + j]; A[piv * 6 + j] = t; }
      const double t = b[k]; b[k] = b[piv]; b[piv] = t;
    }
    for (int i = k + 1; i < 6; ++i) {
      const double f = A[i * 6 + k] / A[k * 6 + k];
      for (int j = k; j < 6; ++j) A[i * 6 + j] -= f * A[k * 6 + j];
      b[i] -= f * b[k];
    }
  }
  for (int i = 5; i >= 0; --i) {
    double s = b[i];
    for (int j = i + 1; j < 6; ++j) s -= A[i * 6 + j] * x[j];
    x[i] = s / A[i * 6 + i];
  }
  return true;
}

__device__ double hyp_cost(const HypArgs& a, const double* G, const int* id, double* r, double* Xc) {
  double c = 0.0;
  for (int m = 0; m < 4; ++m) {
    const int i = id[m];
    const double X = a.pt3d[i], Y = a.pt3d[a.npts + i], Z = a.pt3d[2 * a.npts + i];
    double xc, yc, zc;
    rigid_apply(G, X, Y, Z, xc, yc, zc);
    Xc[3 * m] = xc; Xc[3 * m + 1] = yc; Xc[3 * m + 2] = zc;
    if (!(zc > 1e-12)) return -1.0;
    r[2 * m] = xc / zc * a.fx + a.cx - a.pt2d[i];
    r[2 * m + 1] = yc / zc * a.fy + a.cy - a.pt2d[a.npts + i];
    c += r[2 * m] * r[2 * m] + r[2 * m + 1] * r[2 * m + 1];
  }
  return c;
}

__global__ void k_hyp_solve(const HypArgs a) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= a.nsamples) return;
  int id[4];
  for (int m = 0; m < 4; ++m) id[m] = a.sample[4 * s + m];
  int ok = 1;
  // degenerate sample: a repeated correspondence or three of the four image points (nearly) collinear
  for (int m = 0; m < 4 && ok; ++m)
    for (int n = m + 1; n < 4; ++n)
      if (id[m] == id[n] || id[m] < 0 || id[m] >= a.npts || id[n] < 0 || id[n] >= a.npts) ok = 0;
  for (int m = 0; m < 4 && ok; ++m) {           // leave point m out
    int q[3], k = 0;
    for (int n = 0; n < 4; ++n) if (n != m) q[k++] = id[n];
    const double ax = a.pt2d[q[1]] - a.pt2d[q[0]], ay = a.pt2d[a.npts + q[1]] - a.pt2d[a.npts + q[0]];
    const double bx = a.pt2d[q[2]] - a.pt2d[q[0]], by = a.pt2d[a.npts + q[2]] - a.pt2d[a.npts + q[0]];
    const double area2 = fabs(ax * by - ay * bx), len = sqrt(ax * ax + ay * ay) * sqrt(bx * bx + by * by);
    if (!(area2 > 1e-3 * len)) ok = 0;
  }
  double p[6], G[12];
  for (int k = 0; k < 6; ++k) p[k] = a.p_init[k];
  se3_exp<double>(G, p);
  double r[8], Xc[12], lambda = 1e-4;
  double cost = ok ? hyp_cost(a, G, id, r, Xc) : -1.0;
  if (cost < 0.0) ok = 0;
  for (int it = 0; it < a.maxiter && ok; ++it) {
    double H[36], g[6];
    for (int k = 0; k < 36; ++k) H[k] = 0.0;
    for (int k = 0; k < 6; ++k) g[k] = 0.0;
    for (int m = 0; m < 4; ++m) {
      const double xc = Xc[3 * m], yc = Xc[3 * m + 1], zc = Xc[3 * m + 2], iz = 1.0 / zc;
      // d(u,v)/d(Xc) times d(Xc)/d(xi) with d(Xc)/d(xi) = [I | -[Xc]x]
      const double ju[3] = {a.fx * iz, 0.0, -a.fx * xc * iz * iz}, jv[3] = {0.0, a.fy * iz, -a.fy * yc * iz * iz};
      double J[2][6];
      for (int e = 0; e < 2; ++e) {
        const double* j = e ? jv : ju;
        J[e][0] = j[0]; J[e][1] = j[1]; J[e][2] = j[2];
        J[e][3] = -j[1] * zc + j[2] * yc;        // column of -[Xc]x for w_x: (0, -z, y)
        J[e][4] = j[0] * zc - j[2] * xc;         // w_y: (z, 0, -x)
        J[e][5] = -j[0] * yc + j[1] * xc;        // w_z: (-y, x, 0)
      }
      for (int e = 0; e < 2; ++e)
        for (int i = 0; i < 6; ++i) {
          g[i] += J[e][i] * r[2 * m + e];
          for (int j = 0; j < 6; ++j) H[i * 6 + j] += J[e][i] * J[e][j];
        }
    }
    double A[36], b[6], xi[6];
    for (int k = 0; k < 36; ++k) A[k] = H[k];
    for (int k = 0; k < 6; ++k) { A[k * 6 + k] += lambda * (H[k * 6 + k] + 1e-12); b[k] = -g[k]; }
    if (!hyp_solve6(A, b, xi)) { ok = 0; break; }
    double E[12], Gn[12];
    se3_exp<double>(E, xi);
    for (int rr = 0; rr < 3; ++rr) {
      for (int c = 0; c < 3; ++c) Gn[4 * rr + c] = E[4 * rr] * G[c] + E[4 * rr + 1] * G[4 + c] + E[4 * rr + 2] * G[8 + c];
      Gn[4 * rr + 3] = E[4 * rr] * G[3] + E[4 * rr + 1] * G[7] + E[4 * rr + 2] * G[11] + E[4 * rr + 3];
    }
    double rn[8], Xn[12];
    const double cn = hyp_cost(a, Gn, id, rn, Xn);
    if (cn >= 0.0 && cn <= cost) {
      for (int k = 0; k < 12; ++k) { G[k] = Gn[k]; Xc[k] = Xn[k]; }
      for (int k = 0; k < 8; ++k) r[k] = rn[k];
      const bool done = cost - cn <= 1e-24 + 1e-16 * cost;
      cost = cn;
      lambda = lambda * 0.1 > 1e-12 ? lambda * 0.1 : 1e-12;
      if (done) break;
    } else {
      lambda *= 10.0;
      if (lambda > 1e8) break;
    }
  }
  // a minimal sample that is consistent with a pose reprojects to its four points (8 equations, 6 unknowns)
  if (ok && !(cost <= 4.0 * a.inlthresh * a.inlthresh)) ok = 0;
  se3_log<double>(p, G);
  for (int k = 0; k < 6; ++k) a.pose[6 * s + k] = ok ? p[k] : 0.0;
  a.status[s] = ok;
}

// reprojection of all correspondences with every solved pose; inlier iff the pixel distance <= inlthresh
// (func_ransac_fitcameras_odom.m:48-52); a sample with fewer than 4 inliers is rejected (:53-57)
__global__ void __launch_bounds__(256) k_hyp_inliers(const HypArgs a) {
  const int s = blockIdx.x;
  __shared__ double sG[12];
  __shared__ int s_cnt;
  if (threadIdx.x == 0) {
    double p[6];
    for (int k = 0; k < 6; ++k) p[k] = a.pose[6 * s + k];
    se3_exp<double>(sG, p);
    s_cnt = 0;
  }
  __syncthreads();
  const bool ok = a.status[s] != 0;
  int cnt = 0;
  for (int i = threadIdx.x; i < a.npts; i += blockDim.x) {
    unsigned char in = 0;
    if (ok) {
      const double X = a.pt3d[i], Y = a.pt3d[a.npts + i], Z = a.pt3d[2 * a.npts + i];
      const double xc = sG[0] * X + sG[1] * Y + sG[2] * Z + sG[3], yc = sG[4] * X + sG[5] * Y + sG[6] * Z + sG[7];
      const double zc = sG[8] * X + sG[9] * Y + sG[10] * Z + sG[11];
      if (zc > 1e-12) {
        const double du = xc / zc * a.fx + a.cx - a.pt2d[i], dv = yc / zc * a.fy + a.cy - a.pt2d[a.npts + i];
        in = sqrt(du * du + dv * dv) <= a.inlthresh;
      }
    }
    a.mask[(size_t)s * a.npts + i] = in;
    cnt += in;
  }
  atomicAdd(&s_cnt, cnt);
  __syncthreads();
  if (threadIdx.x == 0) {
    a.ninl[s] = s_cnt;
    if (s_cnt < 4) a.status[s] = 0;
  }
}

cudaError_t launch_hypotheses(const double fc[2], const double cc[2], int npts, const double* pt2d, const double* pt3d,
                              int nsamples, const int* sample, const double p_init[6], double inlthresh, int maxiter,
                              double* pose, int* status, int* ninl, unsigned char* mask, cudaStream_t stream) {
  if (nsamples <= 0) return cudaSuccess;
  HypArgs a;
  a.fx = fc[0]; a.fy = fc[1]; a.cx = cc[0]; a.cy = cc[1];
  a.npts = npts; a.nsamples = nsamples; a.maxiter = maxiter; a.inlthresh = inlthresh;
  a.pt2d = pt2d; a.pt3d = pt3d; a.sample = sample;
  for (int k = 0; k < 6; ++k) a.p_init[k] = p_init[k];
  a.pose = pose; a.status = status; a.ninl = ninl; a.mask = mask;
  k_hyp_solve<<<(nsamples + 127) / 128, 128, 0, stream>>>(a);
  count_launch();
  k_hyp_inliers<<<nsamples, 256, 0, stream>>>(a);
  count_launch();
  return cudaGetLastError();
}

}  // namespace ict
