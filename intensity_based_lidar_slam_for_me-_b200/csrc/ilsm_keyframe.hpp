// ilsm_keyframe.hpp -- the full loop's keyframe rule (ilsm_slam_enable_loop).  Plain C++ with no CUDA or library
// headers, so that a CPU test can build it on its own and hold a restatement to it bit for bit.
#pragma once
#include <math.h>

namespace ilsm {

// Is the frame with mapped pose (q, t) (xyzw, world <- frame) a keyframe, given the last keyframe's (q_kf, t_kf)?  Every
// step is one fp64 operation in the order written (_build.py compiles host code with -ffp-contract=off): the
// distance is sqrt((dx*dx + dy*dy) + dz*dz); (v, w) is the Hamilton product conj(q_kf) * q; the angle 2 atan2(|v|, |w|).
inline bool keyframe_due(const double q_kf[4], const double t_kf[3], const double q[4], const double t[3], double dist,
                         double angle) {
  const double dx = t[0] - t_kf[0], dy = t[1] - t_kf[1], dz = t[2] - t_kf[2];
  const double d = sqrt(dx * dx + dy * dy + dz * dz);
  const double ax = -q_kf[0], ay = -q_kf[1], az = -q_kf[2], aw = q_kf[3];
  const double vx = aw * q[0] + ax * q[3] + ay * q[2] - az * q[1];
  const double vy = aw * q[1] - ax * q[2] + ay * q[3] + az * q[0];
  const double vz = aw * q[2] + ax * q[1] - ay * q[0] + az * q[3];
  const double w = aw * q[3] - ax * q[0] - ay * q[1] - az * q[2];
  const double a = 2.0 * atan2(sqrt(vx * vx + vy * vy + vz * vz), fabs(w));
  return d >= dist || a >= angle;
}

}  // namespace ilsm
