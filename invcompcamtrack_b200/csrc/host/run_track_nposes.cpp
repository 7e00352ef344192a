// run_track_nposes — N pose hypotheses tracked forward and backward over a frame sequence and scored by patch NCC,
// with the text formats of the reference driver (run_track_nposes.cpp:39-131):
//
//   run_track_nposes infile outfile
//   infile   line 1  lv_f lv_l psz maxiter normdp_ratio donorm dopatchnorm maxpttrack verbosity
//            line 2  fx fy cx cy w h          line 3  nback nfwd          then nback+nfwd+1 image names (binary PGM)
//            nocorresp, that many "x y X Y Z";  nosamples, per sample "p0..p5 noids id.." (ids are 1-based)
//   outfile  per sample: one line of 6 values (precision 8) per image, then one line of NCC values (precision 3)
//
// The reference walks the samples one at a time through one OdometerClass (:193-361).  Samples are independent, so
// here they are a BATCH: all forward chains advance together (ict_track_sequence), then all backward chains, then
// one NCC launch; only poses and correlations leave the device.  Two quirks of the reference are kept on purpose:
// its NCC step sets op.dopatchnorm = true and never resets it (:281), so every sample after the first is TRACKED
// with patch normalisation whatever the input file says; and Set3Dpoints runs once per sample, not per frame.
// The reference's summation order (Eigen's 4-float SSE packets) is the default; ICT_SUM_ORDER=3 selects that order with
// 8-float AVX packets (a reference built with -mavx), 0 the fast mode.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iomanip>
#include <iostream>
#include <sstream>
#include <string>
#include <vector>

#include "image_io.h"
#include "utilities.h"

using namespace CTR;

struct Input {
  optparam op;
  float fc[2], cc[2];
  int wh[2], fb[2];
  std::vector<std::string> files;
  std::vector<double> xyz;                 // 3 per correspondence
  std::vector<std::vector<double>> poses;  // 6 per sample
  std::vector<std::vector<int>> ids;
};

static bool read_input(const char* name, Input& in) {
  std::ifstream f(name);
  if (!f) return false;
  int lv_f, lv_l, psz, maxiter, donorm, patchnorm, maxpt, verb;
  float ratio;
  f >> lv_f >> lv_l >> psz >> maxiter >> ratio >> donorm >> patchnorm >> maxpt >> verb;
  ict_optparam_init(&in.op, lv_f, lv_l, psz, maxiter, ratio, donorm, patchnorm, maxpt, verb);
  f >> in.fc[0] >> in.fc[1] >> in.cc[0] >> in.cc[1] >> in.wh[0] >> in.wh[1];
  f >> in.fb[0] >> in.fb[1];
  in.files.resize(in.fb[0] + in.fb[1] + 1);
  for (auto& s : in.files) f >> s;
  int nc = 0;
  f >> nc;
  in.xyz.resize(3 * (size_t)nc);
  for (int i = 0; i < nc; ++i) {
    double x2, y2;
    f >> x2 >> y2 >> in.xyz[3 * i] >> in.xyz[3 * i + 1] >> in.xyz[3 * i + 2];
  }
  int ns = 0;
  f >> ns;
  in.poses.assign(ns, std::vector<double>(6));
  in.ids.resize(ns);
  for (int s = 0; s < ns; ++s) {
    for (int k = 0; k < 6; ++k) f >> in.poses[s][k];
    int n = 0;
    f >> n;
    in.ids[s].resize(n);
    for (int k = 0; k < n; ++k) f >> in.ids[s][k];
  }
  return (bool)f;
}

#define CHECK(call)                                                        \
  do {                                                                     \
    if ((call) != ICT_OK) {                                                \
      std::printf("%s failed: %s\n", #call, ict_last_error());             \
      return 1;                                                            \
    }                                                                      \
  } while (0)

// tracks samples [s0, s1) as one batch; fills out_pose[s][image][6] and out_corr[s][point]
static int run_batch(const Input& in, const optparam& op, ict_frames* fs, int s0, int s1,
                     std::vector<std::vector<std::vector<double>>>& out_pose, std::vector<std::vector<double>>& out_corr) {
  const int T = s1 - s0, nimg = (int)in.files.size(), nb = in.fb[0], nf = in.fb[1];
  std::vector<int64_t> off(T + 1, 0);
  for (int t = 0; t < T; ++t) off[t + 1] = off[t] + (int64_t)in.ids[s0 + t].size();
  const int64_t total = off[T];
  std::vector<double> pts(3 * (size_t)total), p0(6 * (size_t)T);
  for (int t = 0; t < T; ++t) {
    const auto& id = in.ids[s0 + t];
    const size_t n = id.size();
    for (size_t i = 0; i < n; ++i)
      for (int k = 0; k < 3; ++k) pts[3 * off[t] + k * n + i] = in.xyz[3 * (size_t)(id[i] - 1) + k];   // :207-213
    std::copy(in.poses[s0 + t].begin(), in.poses[s0 + t].end(), p0.begin() + 6 * t);
  }
  ict_tracker* tr = ict_tracker_create(&op, in.fc, in.cc, in.wh);
  if (!tr) { std::printf("ict_tracker_create: %s\n", ict_last_error()); return 1; }
  if (const char* so = std::getenv("ICT_SUM_ORDER")) CHECK(ict_tracker_set_sum_order(tr, std::atoi(so)));
  // The reference resets its patch / steepest-descent arrays only in Set3Dpoints (odometer.cpp:173): a point that leaves
  // the image keeps its last template through the rest of the sample's chains.  Reproduced by the tracker's keep_state
  // (reference order, psz 8, <= 224 points); ICT_KEEP_STATE=0 turns it off (every frame step then starts from zero).
  int keep = std::getenv("ICT_KEEP_STATE") ? std::atoi(std::getenv("ICT_KEEP_STATE")) : 1;
  CHECK(ict_tracker_set_knob(tr, "keep_state", keep));
  CHECK(ict_tracker_set_points(tr, T, off.data(), pts.data(), 0));

  std::vector<float> q_ref(2 * (size_t)total), q_fwd(2 * (size_t)total), q_back(2 * (size_t)total), corr((size_t)total);
  CHECK(ict_tracker_reproject(tr, p0.data(), q_ref.data()));                                       // :217-225
  std::vector<double> fwd(6 * (size_t)T * (nf + 1)), back(6 * (size_t)T * (nb + 1));
  int rc_seq = ict_track_sequence(tr, fs, nb, nf, +1, p0.data(), fwd.data(), nullptr, nullptr);   // :232-239
  if (rc_seq == ICT_ERR_UNSUPPORTED && keep) {
    std::printf("note: this configuration runs without the reference's state between frame steps (%s)\n", ict_last_error());
    keep = 0;
    CHECK(ict_tracker_set_knob(tr, "keep_state", 0));
    rc_seq = ict_track_sequence(tr, fs, nb, nf, +1, p0.data(), fwd.data(), nullptr, nullptr);
  }
  CHECK(rc_seq);
  CHECK(ict_tracker_reproject(tr, fwd.data() + 6 * (size_t)T * nf, q_fwd.data()));                 // :240-246
  CHECK(ict_track_sequence(tr, fs, nb, nb, -1, p0.data(), back.data(), nullptr, nullptr));         // :250-258
  CHECK(ict_tracker_reproject(tr, back.data() + 6 * (size_t)T * nb, q_back.data()));               // :259-265
  CHECK(ict_ncc_score(tr, fs, 0, nb, nimg - 1, nb, nf, q_back.data(), q_ref.data(), q_fwd.data(), corr.data()));
  for (int t = 0; t < T; ++t) {
    auto& po = out_pose[s0 + t];
    po.assign(nimg, std::vector<double>(6, 0.0));
    for (int k = 0; k <= nf; ++k) std::copy_n(fwd.begin() + 6 * ((size_t)k * T + t), 6, po[nb + k].begin());
    for (int k = 1; k <= nb; ++k) std::copy_n(back.begin() + 6 * ((size_t)k * T + t), 6, po[nb - k].begin());
    out_corr[s0 + t].assign(corr.begin() + off[t], corr.begin() + off[t + 1]);
  }
  ict_tracker_destroy(tr);
  return 0;
}

int main(int argc, char** argv) {
  if (argc < 3) {
    std::printf("usage: %s infile outfile\n", argv[0]);
    return 2;
  }
  Input in;
  if (!read_input(argv[1], in)) {
    std::printf("could not parse %s\n", argv[1]);
    return 1;
  }
  const int nimg = (int)in.files.size(), ns = (int)in.poses.size();
  ict_frames* fs = ict_frames_create(nimg, in.wh[0], in.wh[1], in.op.lv_f, in.op.psz);
  if (!fs) { std::printf("ict_frames_create: %s\n", ict_last_error()); return 1; }
  for (int i = 0; i < nimg; ++i) {   // imread + util_constructpyramide for every frame, :160-181
    std::vector<unsigned char> pix;
    int w = 0, h = 0;
    if (!ictio::read_pgm(in.files[i], pix, w, h) || w != in.wh[0] || h != in.wh[1]) {
      std::printf("could not read %s as a %dx%d binary PGM\n", in.files[i].c_str(), in.wh[0], in.wh[1]);
      return 1;
    }
    CHECK(ict_frames_upload_u8(fs, i, 1, pix.data()));
  }
  std::vector<std::vector<std::vector<double>>> out_pose(ns);
  std::vector<std::vector<double>> out_corr(ns);
  if (ns > 0) {
    if (run_batch(in, in.op, fs, 0, 1, out_pose, out_corr)) return 1;
    if (ns > 1) {
      optparam op2 = in.op;
      op2.dopatchnorm = 1;   // the reference never resets it after the first sample's NCC step (:281)
      if (run_batch(in, op2, fs, 1, ns, out_pose, out_corr)) return 1;
    }
  }
  std::ofstream out(argv[2]);   // WriteResult, :106-131
  for (int s = 0; s < ns; ++s) {
    out << std::setprecision(8);
    for (const auto& p : out_pose[s]) {
      for (int k = 0; k < 6; ++k) out << p[k] << " ";
      out << std::endl;
    }
    out << std::setprecision(3);
    for (double c : out_corr[s]) out << c << " ";
    out << std::endl;
  }
  ict_frames_destroy(fs);
  return 0;
}
