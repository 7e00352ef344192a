// run_track — single-pair tracker with the command line and file formats of the reference's working single-pair
// driver (run_io_reprojection_test.cpp:99-235; the reference's own run_track.cpp is a non-compiling stub of it):
//
//   run_track imgA imgB infile outfile lv_f lv_l psz maxiter normdp_ratio donorm dopatchnorm maxpttrack verbosity
//
//   infile  (binary, little endian)  6 f64 pose | 2 f32 fc | 2 f32 cc | 2 u32 wh | u64 N | N f64 X | N f64 Y | N f64 Z |
//                                    N f32 x2d | N f32 y2d                        (run_io_reprojection_test.cpp:54-79)
//   outfile (binary)                 6 f64 pose                                   (:83-97)
//   images  binary PGM (P5) instead of whatever cv::imread accepts.
// Written against the reference's class interface (CamClass / PoseClass / OdometerClass / util_constructpyramide);
// the alignment itself runs on the GPU.  The reference's summation order (Eigen's 4-float SSE packets) is the default;
// ICT_SUM_ORDER=3 selects that order with 8-float AVX packets (a reference built with -mavx), 0 the fast mode.
#include <sys/time.h>

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "camera.h"
#include "image_io.h"
#include "odometer.h"
#include "pose.h"
#include "utilities.h"

using namespace CTR;

static bool read_input(const char* name, double pose[6], float fc[2], float cc[2], int wh[2], std::vector<double>& xyz,
                       int& n) {
  FILE* f = std::fopen(name, "rb");
  if (!f) return false;
  uint32_t whu[2];
  uint64_t cnt = 0;
  bool ok = std::fread(pose, sizeof(double), 6, f) == 6 && std::fread(fc, sizeof(float), 2, f) == 2 &&
            std::fread(cc, sizeof(float), 2, f) == 2 && std::fread(whu, sizeof(uint32_t), 2, f) == 2 &&
            std::fread(&cnt, sizeof(uint64_t), 1, f) == 1;
  if (ok) {
    n = (int)cnt;
    wh[0] = (int)whu[0];
    wh[1] = (int)whu[1];
    xyz.resize(3 * (size_t)n);   // X block, Y block, Z block: what Set3Dpoints expects
    ok = std::fread(xyz.data(), sizeof(double), 3 * (size_t)n, f) == 3 * (size_t)n;
  }
  std::fclose(f);
  return ok;
}

int main(int argc, char** argv) {
  if (argc < 14) {
    std::printf("usage: %s imgA imgB infile outfile lv_f lv_l psz maxiter normdp_ratio donorm dopatchnorm maxpttrack "
                "verbosity\n", argv[0]);
    return 2;
  }
  optparam op;
  ict_optparam_init(&op, std::atoi(argv[5]), std::atoi(argv[6]), std::atoi(argv[7]), std::atoi(argv[8]),
                    (float)std::atof(argv[9]), std::atoi(argv[10]), std::atoi(argv[11]), std::atoi(argv[12]),
                    std::atoi(argv[13]));

  cv::Mat img[2];
  for (int k = 0; k < 2; ++k) {
    std::vector<unsigned char> pix;
    int w = 0, h = 0;
    if (!ictio::read_pgm(argv[1 + k], pix, w, h)) {
      std::printf("could not read %s (binary PGM expected)\n", argv[1 + k]);
      return 1;
    }
    img[k].create(h, w, CV_8U);
    std::memcpy(img[k].data, pix.data(), pix.size());
  }

  double p_in[6], p_out[6] = {0, 0, 0, 0, 0, 0};
  float fc[2], cc[2];
  int wh[2], n = 0;
  std::vector<double> xyz;
  if (!read_input(argv[3], p_in, fc, cc, wh, xyz, n)) {
    std::printf("ReadFile: could not read %s\n", argv[3]);
    return 1;
  }

  const int L = op.lv_f + 1;
  std::vector<cv::Mat> a(L), adx(L), ady(L), b(L), bdx(L), bdy(L);
  std::vector<const float*> pa(L), pax(L), pay(L), pb(L), pbx(L), pby(L);
  util_constructpyramide(img[0], a.data(), adx.data(), ady.data(), pa.data(), pax.data(), pay.data(), op.lv_f, 1, op.psz);
  util_constructpyramide(img[1], b.data(), bdx.data(), bdy.data(), pb.data(), pbx.data(), pby.data(), op.lv_f, 1, op.psz);

  const CamClass cam(op.lv_f + 1, fc, cc, wh, op.psz);
  PoseClass pose(&cam, &op);
  OdometerClass odom(&pose, &op);
  if (const char* so = std::getenv("ICT_SUM_ORDER")) odom.SetSumOrder(std::atoi(so));

  timeval t0, t1;
  gettimeofday(&t0, nullptr);
  const int reps = op.verbosity == 1 ? 1000 : 1;   // the reference times 1000 repetitions (:209-218)
  for (int r = 0; r < reps; ++r) {
    odom.Set3Dpoints(xyz.data(), n);
    odom.SetPose(p_in, pa.data(), pax.data(), pay.data(), pb.data());
    odom.TrackPose(p_out);
  }
  gettimeofday(&t1, nullptr);
  if (op.verbosity == 1)
    std::printf("TIME (pose tracking) (musec): %3g\n", (t1.tv_sec - t0.tv_sec) * 1000.0 + (t1.tv_usec - t0.tv_usec) / 1000.0);
  if (op.verbosity == 2) {
    const int* it = odom.LastIterations();
    for (int l = 0; l <= op.lv_f - op.lv_l; ++l) std::printf("Sc%02i: %d iterations\n", op.lv_f - l, it[l]);
  }

  FILE* f = std::fopen(argv[4], "wb");
  if (!f || std::fwrite(p_out, sizeof(double), 6, f) != 6) std::printf("WriteFile: problem writing %s\n", argv[4]);
  if (f) std::fclose(f);
  util_release_device_pyramids();
  return 0;
}
