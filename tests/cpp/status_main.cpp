/* Drives ekfcuda::Robot::localize (include/ekf_robot.hpp) through both exceptional statuses: a scan whose first fit
 * skips a singular pair (EKF_ESINGULAR) and a scan with more new lines than free slots (EKF_ECAPACITY).  Neither may
 * throw, and lastStatus must hold the code.  The filter's heading has zero variance at rest (zero odometry), so a
 * landmark appended from a line with R00 = R01 = 0 has an angle of zero variance and S is exactly singular with every
 * such line.  Built and run by tests/test_gpu_exceptional.py; prints "status_main OK" when every check holds. */
#include <cstdio>
#include <vector>
#include "ekf_robot.hpp"

struct Mat { double* data; };
struct PolarPoint { double alfa, r; };
struct Line { double alfa, r; Mat* C_AR; std::vector<PolarPoint> lineInterval; };

#define CHECK(c) do { if (!(c)) { std::printf("FAILED: %s (line %d)\n", #c, __LINE__); return 1; } } while (0)

int main() {
  double reg[4] = {4e-6, 0.0, 0.0, 2.5e-5}, sing[4] = {0.0, 0.0, 0.0, 2.5e-5};
  Mat mr = {reg}, ms = {sing};
  const double enc[3] = {0.0, 0.0, 0.0};             /* at rest: zero odometry */
  ekfcuda::Robot rover(0, 0, 0, 13);                 /* the map resets above 13 - 10 landmarks */
  std::vector<Line> a(2);
  a[0].alfa = 0.0; a[0].r = 2.0; a[0].C_AR = &ms;
  a[1].alfa = 1.0; a[1].r = 3.0; a[1].C_AR = &mr;
  rover.localize(a, (float*)0, enc);
  CHECK(rover.lastStatus == EKF_OK && rover.savedLineCount == 2);
  std::vector<Line> b(1);                            /* singular with landmark 0, then matches landmark 1 */
  b[0].alfa = 1.0; b[0].r = 3.0; b[0].C_AR = &ms;
  rover.localize(b, (float*)0, enc);
  CHECK(rover.lastStatus == EKF_ESINGULAR && rover.lastMatches[0] == 1 && rover.savedLineCount == 2);
  std::vector<Line> c(12);                           /* 12 new lines, 11 free slots: one dropped, then the reset */
  for (int i = 0; i < 12; ++i) { c[i].alfa = -3.0 + 0.4 * i; c[i].r = 5.0 + 0.2 * i; c[i].C_AR = &mr; }
  rover.localize(c, (float*)0, enc);
  CHECK(rover.lastStatus == EKF_ECAPACITY && rover.savedLineCount == 0);
  rover.localize(b, (float*)0, enc);                 /* the empty map: appended, a clean scan */
  CHECK(rover.lastStatus == EKF_OK && rover.savedLineCount == 1);
  std::printf("status_main OK\n");
  return 0;
}
