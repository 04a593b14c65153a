/* Drives ekfcuda::Robot::observePose (include/ekf_robot.hpp): a map of ten walls seen from a robot at rest, then an
 * absolute fix that moves the pose.  The mirrors must follow the fix (localize predicts from them), a tight gate must
 * reject a far fix without changing anything, and a singular fix (theta alone with R_thth = 0 on a fresh filter) must
 * leave the state as it was.  Built and run by tests/test_gpu_pose_fix.py; prints "pose_fix_main OK" when every check
 * holds. */
#include <cmath>
#include <cstdio>
#include <stdexcept>
#include <vector>
#include "ekf_robot.hpp"

struct Mat { double* data; };
struct PolarPoint { double alfa, r; };
struct Line { double alfa, r; Mat* C_AR; std::vector<PolarPoint> lineInterval; };

#define CHECK(c) do { if (!(c)) { std::printf("FAILED: %s (line %d)\n", #c, __LINE__); return 1; } } while (0)

int main() {
  {
    ekfcuda::Robot fresh(0, 0, 0, 20);
    const double z[3] = {0.0, 0.0, 0.3}, R[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    CHECK(!fresh.observePose(z, R, EKF_POSE_THETA));
    CHECK(fresh.xPos == 0.0 && fresh.yPos == 0.0 && fresh.thetaPos == 0.0);
  }
  ekfcuda::Robot rover(0, 0, 0, 200);
  double cov[4] = {4e-6, 0.0, 0.0, 2.5e-5};
  Mat m = {cov};
  std::vector<Line> walls(10);
  for (int i = 0; i < 10; ++i) {
    walls[i].alfa = -3.0 + 0.6 * i;
    walls[i].r = 2.0 + 0.4 * i;
    walls[i].C_AR = &m;
  }
  const double enc[3] = {0.0, 0.0, 0.0};             /* at rest: (pose - encoder) = 0 */
  rover.localize(walls, (float*)0, enc);
  rover.localize(walls, (float*)0, enc);
  CHECK(rover.savedLineCount == 10);
  const double far[3] = {5.0, 5.0, 1.0}, R[9] = {1e-4, 0, 0, 0, 1e-4, 0, 0, 0, 1e-4};
  double d2 = -1.0;
  CHECK(!rover.observePose(far, R, EKF_POSE_X | EKF_POSE_Y | EKF_POSE_THETA, 11.34, &d2));   /* chi2(3) at 0.99 */
  CHECK(d2 > 11.34 && rover.xPos == 0.0 && rover.yPos == 0.0);
  const double fix[3] = {0.01, -0.02, 0.005};
  CHECK(rover.observePose(fix, R, EKF_POSE_X | EKF_POSE_Y | EKF_POSE_THETA, HUGE_VAL, &d2));
  CHECK(d2 >= 0.0 && rover.xPos > 0.0 && rover.yPos < 0.0);   /* theta stays: at rest P[2,2] = 0 (no motion noise) */
  double pose[3];
  ekf_get_state(rover.context(), pose, 0, 0);
  CHECK(pose[0] == rover.xPos && pose[1] == rover.yPos && pose[2] == rover.thetaPos);
  const double xb = rover.xPos;
  const double enc2[3] = {rover.xPos, rover.yPos, rover.thetaPos};   /* no motion since the fix: u = 0 */
  rover.localize(walls, (float*)0, enc2);
  for (int i = 0; i < 10; ++i) CHECK(rover.lastMatches[i] == i);
  CHECK(std::fabs(rover.xPos - xb) < 0.01);
  bool threw = false;
  try { rover.observePose(fix, R, 0); } catch (const std::runtime_error&) { threw = true; }
  CHECK(threw);
  std::printf("pose_fix_main OK\n");
  return 0;
}
