// odometer.h — OdometerClass with the reference's interface (odometer.h:18-116): Set3Dpoints / SetPose / TrackPose /
// Get2DPoints.  Every call forwards to the device-side tracker of libictrack.so (one track per object, as in the
// reference); batches of tracks should use the C ABI directly (ict_track_batch).
#ifndef ICT_HOST_ODOMETER_HEADER
#define ICT_HOST_ODOMETER_HEADER

#include <vector>

#include "camera.h"
#include "pose.h"
#include "utilities.h"

namespace CTR {

class OdometerClass {
 public:
  OdometerClass(PoseClass* pose_in, const optparam* op_in);
  ~OdometerClass();

  void Set3Dpoints(double* pt_in, const int nopoints_in);
  void SetPose(const double* p_in, const float** img_ref_in, const float** img_ref_dx_in, const float** img_ref_dy_in,
               const float** img_new_in);
  void TrackPose(double* p_out);
  inline const float* Get2DPoints() const { return pt2d_lvl.data(); }   // x block, y block at stride maxpttrack

  // not in the reference: iterations run per level by the last TrackPose (coarse to fine), -1 before the first call
  inline const int* LastIterations() const { return iters; }
  // the order of the fp32 sums (ict_tracker_set_sum_order): 1 (default) the reference's order with Eigen's 4-float SSE
  // packets, 3 with its 8-float AVX packets (a reference built with -mavx), 0 fast tree reductions
  void SetSumOrder(int mode);

 private:
  bool bind_frame(int slot, const float** I, const float** dx, const float** dy);
  PoseClass* pose;
  const optparam* op;
  ict_tracker* tracker;
  ict_frames* view;       // two aliases: 0 = reference frame, 1 = new frame
  ict_frames* scratch;    // holds planes this library did not build itself
  int nopoints, n_in;
  double p_cur[6];
  int iters[ICT_MAX_LEVELS];
  std::vector<float> pt2d_lvl;
};

}  // namespace CTR
#endif
