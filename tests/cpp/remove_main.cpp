/* Drives ekfcuda::Robot::removeLines (include/ekf_robot.hpp): a map of ten walls seen from a robot at rest, three of
 * them removed, then the next localize re-appends exactly those three.  Built and run by tests/test_gpu_remove_lines.py;
 * prints "remove_main OK" when every check holds. */
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
  CHECK(rover.savedLineCount == 10);
  rover.localize(walls, (float*)0, enc);
  CHECK(rover.savedLineCount == 10);
  for (int i = 0; i < 10; ++i) CHECK(rover.lastMatches[i] == i);
  CHECK(rover.removeLines(std::vector<int>{0, 3, 7}) == 7);
  CHECK(rover.savedLineCount == 7);
  CHECK(rover.removeLines(std::vector<int>()) == 7);
  bool threw = false;
  try { rover.removeLines(std::vector<int>{2, 1}); } catch (const std::runtime_error&) { threw = true; }
  CHECK(threw && rover.savedLineCount == 7);
  rover.localize(walls, (float*)0, enc);
  CHECK(rover.savedLineCount == 10);
  const int expect[10] = {-1, 0, 1, -1, 2, 3, 4, -1, 5, 6};   /* kept walls moved down in order; removed ones re-appended */
  for (int i = 0; i < 10; ++i) CHECK(rover.lastMatches[i] == expect[i]);
  rover.localize(walls, (float*)0, enc);
  const int again[10] = {7, 0, 1, 8, 2, 3, 4, 9, 5, 6};
  for (int i = 0; i < 10; ++i) CHECK(rover.lastMatches[i] == again[i]);
  CHECK(std::fabs(rover.xPos) < 1e-6 && std::fabs(rover.yPos) < 1e-6);
  std::printf("remove_main OK\n");
  return 0;
}
