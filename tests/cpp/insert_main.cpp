/* Drives ekfcuda::Robot::insertLines (include/ekf_robot.hpp): ten surveyed walls inserted before the first localize of a
 * robot at rest; every line then matches them and nothing is appended.  Errors throw and leave savedLineCount; the map
 * reset drops the walls with the rest of the map, and they go back in.  Built and run by tests/test_gpu_insert_lines.py;
 * prints "insert_main OK" when every check holds. */
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
  ekfcuda::Robot rover(0, 0, 0, 200);                /* capacity 200, the reference's reset headroom of 10 */
  double cov[4] = {4e-6, 0.0, 0.0, 2.5e-5};
  Mat m = {cov};
  std::vector<Line> walls(10);
  std::vector<double> plan;
  for (int i = 0; i < 10; ++i) {
    walls[i].alfa = -3.0 + 0.6 * i;
    walls[i].r = 2.0 + 0.4 * i;
    walls[i].C_AR = &m;
    plan.push_back(walls[i].alfa);                   /* at the origin the robot frame is the world frame */
    plan.push_back(walls[i].r);
  }
  CHECK(rover.insertLines(plan) == 10);
  CHECK(rover.savedLineCount == 10);
  const double enc[3] = {0.0, 0.0, 0.0};             /* at rest: (pose - encoder) = 0 */
  for (int k = 0; k < 3; ++k) {
    rover.localize(walls, (float*)0, enc);
    CHECK(rover.savedLineCount == 10);
    for (int i = 0; i < 10; ++i) CHECK(rover.lastMatches[i] == i);
  }
  CHECK(std::fabs(rover.xPos) < 1e-6 && std::fabs(rover.yPos) < 1e-6);
  bool threw = false;
  try { rover.insertLines(std::vector<double>{1.0, 2.0, 3.0}); } catch (const std::exception&) { threw = true; }
  CHECK(threw && rover.savedLineCount == 10);
  std::vector<double> far;
  for (int i = 0; i < 191; ++i) { far.push_back(-3.0 + 0.03 * i); far.push_back(50.0 + i); }
  threw = false;
  try { rover.insertLines(far); } catch (const std::runtime_error&) { threw = true; }   /* 201 > 200: nothing inserted */
  CHECK(threw && rover.savedLineCount == 10);
  double bad[4] = {1e-4, 1e-5, 2e-5, 1e-4};                                               /* not symmetric */
  threw = false;
  try { rover.insertLines(std::vector<double>{0.5, 3.0}, bad); } catch (const std::runtime_error&) { threw = true; }
  CHECK(threw && rover.savedLineCount == 10);
  double prior[4] = {1e-4, 1e-5, 1e-5, 1e-4};
  CHECK(rover.insertLines(std::vector<double>{0.5, 30.0}, prior) == 11);
  far.resize(2 * 179);
  CHECK(rover.insertLines(far) == 190);
  /* one line 3 m beyond wall 0 matches nothing and is appended: 191 > 200 - 10 resets the map (Robot.cpp:893-904) */
  std::vector<Line> ghost(1, walls[0]);
  ghost[0].r += 3.0;
  rover.localize(ghost, (float*)0, enc);
  CHECK(rover.savedLineCount == 0);
  CHECK(rover.insertLines(plan) == 10);
  rover.localize(walls, (float*)0, enc);
  CHECK(rover.savedLineCount == 10);
  for (int i = 0; i < 10; ++i) CHECK(rover.lastMatches[i] == i);
  std::printf("insert_main OK\n");
  return 0;
}
