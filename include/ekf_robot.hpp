/* ekf_robot.hpp -- C++ host side of the drop-in: the reference's `Robot` surface over libekfcuda.
 *
 * slam_ros/Robot.h:21-77 declares the class the node uses (slam_ros/main.cpp:98, 144-174):
 *     Robot(double x, double y, double theta);
 *     void localize(const std::vector<line>& lines, float* rot = NULL, const double* encoder = NULL);
 *     bool getEllipse(float axii[2], float& angle);
 *     double xPos, yPos, thetaPos;   double P_t0[SLAMSIZE*SLAMSIZE];   std_msgs::Float32MultiArray lineIntervals;
 *
 * This header provides the same members with the same meaning; every gsl_blas_dgemm of Robot::localize
 * (Robot.cpp:242-860) is replaced by calls into the C ABI of include/ekf.h.  It is a template on the line
 * type so that it compiles against the reference's own `line` (simplifyPath.h:62-79: .alfa, .r,
 * .C_AR->data[4], .lineInterval) inside the catkin package, and against any struct with those members in
 * tests -- no GSL or ROS header is needed here.  INTEGRATION.md shows the two-line change to the node.
 *
 * What stays on the host is exactly what the reference also does outside GSL: the odometry vector from
 * (pose - encoder) (Robot.cpp:135-145, SIMULATIONOFF branch) and the float end points of newly added
 * lines (Robot.cpp:869-879).  P_t0 is NOT mirrored every step (it lives in HBM); syncCovariance() copies it
 * back in the reference's layout when a consumer really wants the whole matrix.
 */
#ifndef LIBEKFCUDA_EKF_ROBOT_HPP
#define LIBEKFCUDA_EKF_ROBOT_HPP

#include <cmath>
#include <cstddef>
#include <stdexcept>
#include <string>
#include <vector>

#include "ekf.h"

namespace ekfcuda {

#ifndef EKF_ROBOT_LINESIZE
#define EKF_ROBOT_LINESIZE 100     /* Robot.h:13 */
#endif

struct FloatArray { std::vector<float> data; };   /* stands in for std_msgs::Float32MultiArray::data (Robot.h:59) */

class Robot {
 public:
  double xPos, yPos, thetaPos;                    /* Robot.h:54-56 */
  FloatArray lineIntervals;                       /* Robot.h:59 */
  std::vector<double> P_t0;                       /* Robot.h:62, filled by syncCovariance() */
  std::vector<double> y;                          /* Robot.h:26, filled by syncCovariance() */
  int savedLineCount;                             /* Robot.h:28, refreshed after every localize */
  std::vector<int> lastMatches;                   /* matched landmark (or -1) per line of the last scan */
  int lastStatus;

  Robot(double x, double yy, double theta, int linesize = EKF_ROBOT_LINESIZE, int device = 0)
      : xPos(x), yPos(yy), thetaPos(theta), savedLineCount(0), lastStatus(EKF_OK), ctx_(0) {
    ekf_config cfg;
    ekf_default_config(&cfg);
    cfg.capacity_lines = linesize;
    cfg.device = device;
    const int rc = ekf_create(&ctx_, &cfg);
    if (rc != EKF_OK) {
      std::string msg = ctx_ ? ekf_last_error(ctx_) : "ekf_create failed";
      if (ctx_) ekf_destroy(ctx_);
      ctx_ = 0;
      throw std::runtime_error("libekfcuda: " + msg);
    }
    n_ = 3 + 2 * linesize;
    lineIntervals.data.reserve(80);               /* Robot.cpp:31 */
  }
  ~Robot() { if (ctx_) ekf_destroy(ctx_); }
  Robot(const Robot&) = delete;
  Robot& operator=(const Robot&) = delete;

  /* Robot::localize (Robot.cpp:126-943).  `rot` is accepted and ignored exactly as the reference does
   * when SIMULATIONOFF is true (Robot.cpp:136-145). */
  template <class Line>
  void localize(const std::vector<Line>& lines, float* rot = 0, const double* encoder = 0) {
    (void)rot;
    if (!encoder) throw std::invalid_argument("Robot::localize: encoder pose required (Robot.cpp:141-143 dereferences it)");
    const double x_t0[3] = {xPos, yPos, thetaPos};                       /* Robot.cpp:130 */
    double u[3] = {0, 0, 0};
    u[2] = x_t0[2] - encoder[2];                                         /* Robot.cpp:141-144 */
    const double dX = x_t0[0] - encoder[0], dY = x_t0[1] - encoder[1];
    u[0] = std::sqrt(dX * dX + dY * dY);
    const int m = (int)lines.size();
    z_.resize(2 * (size_t)m); R_.resize(4 * (size_t)m); lastMatches.assign((size_t)m, -1);
    for (int i = 0; i < m; ++i) {
      z_[2 * i] = lines[i].alfa; z_[2 * i + 1] = lines[i].r;
      for (int t = 0; t < 4; ++t) R_[4 * i + t] = (double)lines[i].C_AR->data[t];   /* Robot.cpp:301-304 with the R[j] fix (Q1) */
    }
    const int L_before = savedLineCount;
    double pose[3];
    lastStatus = ekf_scan(ctx_, x_t0, u, m, m ? z_.data() : 0, m ? R_.data() : 0, m ? lastMatches.data() : 0, pose);
    if (lastStatus != EKF_OK && lastStatus != EKF_ECAPACITY && lastStatus != EKF_ESINGULAR)
      throw std::runtime_error(std::string("libekfcuda: ") + ekf_last_error(ctx_));
    xPos = pose[0]; yPos = pose[1]; thetaPos = pose[2];
    ekf_get_state(ctx_, 0, &savedLineCount, 0);
    /* STORING LINE INTERVALS (Robot.cpp:869-879) for every line that was appended to the map */
    int room = EKF_ROBOT_LINESIZE_ROOM(L_before);
    for (int i = 0; i < m && room > 0; ++i) {
      if (lastMatches[i] >= 0) continue;
      --room;
      if (lines[i].lineInterval.size() == 2) {
        push_endpoint(lines[i].lineInterval.front().alfa, lines[i].lineInterval.front().r);
        push_endpoint(lines[i].lineInterval.back().alfa, lines[i].lineInterval.back().r);
      }
    }
  }

  /* Robot::getEllipse (Robot.cpp:73-124) */
  bool getEllipse(float axii[2], float& angle) {
    int ok = 0;
    if (ekf_get_ellipse(ctx_, axii, &angle, &ok) != EKF_OK) return false;
    return ok != 0;
  }

  /* The `robotPosition` message of the node (slam_ros/main.cpp:150-169): translation = (x, y, theta),
   * rotation.x / .y / .z = major axis, minor axis, angle of the 95 % ellipse.  Plain doubles: the caller
   * copies them into geometry_msgs::Transform. */
  struct RobotPosition { double tx, ty, tz, rx, ry, rz; bool ellipse_ok; };
  RobotPosition robotPosition() {
    RobotPosition msg = {xPos, yPos, thetaPos, 0.0, 0.0, 0.0, false};
    float axii[2] = {0.f, 0.f}, angle = 0.f;
    msg.ellipse_ok = getEllipse(axii, angle);
    msg.rx = axii[1]; msg.ry = axii[0]; msg.rz = angle;
    return msg;
  }

  /* Not in the reference: removes landmarks `lines` (strictly increasing, each below savedLineCount) from the map
   * (ekf_remove_lines) and updates savedLineCount.  A node can prune spurious or long-unseen landmarks with it instead of
   * waiting for the reset of Robot.cpp:893-904.  lineIntervals is the per-scan log the node clears after publishing:
   * untouched.  Returns the new savedLineCount; throws on a bad list. */
  int removeLines(const std::vector<int>& lines) {
    const int rc = ekf_remove_lines(ctx_, (int)lines.size(), lines.empty() ? 0 : lines.data(), &savedLineCount);
    if (rc != EKF_OK) throw std::runtime_error(std::string("libekfcuda: ") + ekf_last_error(ctx_));
    return savedLineCount;
  }

  /* Not in the reference: appends known landmarks (ekf_insert_lines) and updates savedLineCount.  lines = k x (alfa, r)
   * in the world frame, flattened; cov = NULL for surveyed walls (fixed from then on), else the 2k x 2k row-major joint
   * covariance of an earlier map.  Insert a floor plan before the first localize (first fit takes the lowest index), and
   * again after a map reset drops it.  Returns the new savedLineCount; throws on bad input or when the map would exceed
   * its capacity (nothing is inserted then). */
  int insertLines(const std::vector<double>& lines, const double* cov = nullptr) {
    if (lines.size() % 2) throw std::invalid_argument("libekfcuda: insertLines needs (alfa, r) pairs");
    const int rc = ekf_insert_lines(ctx_, (int)(lines.size() / 2), lines.empty() ? 0 : lines.data(), cov, &savedLineCount);
    if (rc != EKF_OK) throw std::runtime_error(std::string("libekfcuda: ") + ekf_last_error(ctx_));
    return savedLineCount;
  }

  /* Not in the reference: fuses an absolute pose measurement (ekf_observe_pose): z = (x, y, theta), R its row-major 3x3
   * covariance, mask of EKF_POSE_X | EKF_POSE_Y | EKF_POSE_THETA (only the selected entries are read), accepted iff S
   * is nonsingular and d2 <= d2Max.  xPos / yPos / thetaPos follow the corrected pose: localize passes them as x_t0
   * (Robot.cpp:130), so a stale mirror would undo the fix at the next prediction.  As after any update, the next localize
   * forms its odometry from the corrected pose and the encoder pose (Robot.cpp:140-145).  Returns whether the fix was
   * accepted (d2 nullable); a singular S returns false with the state unchanged; throws on bad arguments. */
  bool observePose(const double z[3], const double R[9], int mask = EKF_POSE_X | EKF_POSE_Y | EKF_POSE_THETA,
                   double d2Max = HUGE_VAL, double* d2 = 0) {
    int accepted = 0;
    double pose[3];
    const int rc = ekf_observe_pose(ctx_, mask, z, R, d2Max, d2, &accepted, pose);
    if (rc != EKF_OK && rc != EKF_ESINGULAR) throw std::runtime_error(std::string("libekfcuda: ") + ekf_last_error(ctx_));
    xPos = pose[0]; yPos = pose[1]; thetaPos = pose[2];
    return accepted != 0;
  }

  /* copies y and P_t0 back in the reference's layout (SLAMSIZE and SLAMSIZE^2 doubles) */
  void syncCovariance() {
    y.assign((size_t)n_, 0.0); P_t0.assign((size_t)n_ * n_, 0.0);
    ekf_download(ctx_, y.data(), P_t0.data(), &savedLineCount);
  }

  ekf_ctx* context() { return ctx_; }

 private:
  int EKF_ROBOT_LINESIZE_ROOM(int L_before) const { const int cap = (n_ - 3) / 2; return cap > L_before ? cap - L_before : 0; }
  void push_endpoint(double alfa_d, double r) {
    const float alpha = (float)alfa_d;                                    /* `float alpha`, Robot.cpp:871 */
    const double rad = r + xPos * std::cos(alpha) + yPos * std::sin(alpha);   /* cos(float) -> float, as in the reference */
    /* polar_point(alfa, r) scales alfa by PI/180 with PI = 3.14159265 (lineFitting.cpp:71-77): reproduced */
    const double a = ((double)alpha + thetaPos) * (3.14159265 / 180);
    lineIntervals.data.push_back((float)(std::cos(a) * rad));             /* polar2descart, lineFitting.cpp:170-176 */
    lineIntervals.data.push_back((float)(std::sin(a) * rad));
  }
  ekf_ctx* ctx_;
  int n_;
  std::vector<double> z_, R_;
};

/* The device form of what `mapping_cb` does with one `mappingPoints` payload (slam_ros/main.cpp:37-71):
 *     points from (r, angle) float pairs -> lines = LineExtraction(points) -> lin.alfa += M_PI (wrapped).
 * `extract` fills any line type that has the reference's members (simplifyPath.h:62-79): .alfa, .r,
 * .C_AR->data[0..3] and .lineInterval (two {alfa, r} entries).  The reference allocates C_AR with
 * gsl_matrix_alloc(2, 2) inside Covariancia (lineFitting.cpp:384); here the caller passes the allocator
 * (e.g. `[]{ return gsl_matrix_alloc(2, 2); }`), so ownership stays where the node expects it. */
class LineExtractor {
 public:
  explicit LineExtractor(int device = 0, int max_lines = 128) : lx_(0), max_lines_(max_lines), rows_(10 * (size_t)max_lines) {
    const int rc = ekf_lx_create(&lx_, device, max_lines);
    if (rc != EKF_OK) {
      std::string msg = lx_ ? ekf_lx_last_error(lx_) : "ekf_lx_create failed";
      if (lx_) ekf_lx_destroy(lx_);
      lx_ = 0;
      throw std::runtime_error("libekfcuda: " + msg);
    }
  }
  ~LineExtractor() { if (lx_) ekf_lx_destroy(lx_); }
  LineExtractor(const LineExtractor&) = delete;
  LineExtractor& operator=(const LineExtractor&) = delete;

  /* data = msg.data, n_floats = msg.layout.dim[0].size (main.cpp:46).  Appends to `lines`; returns the count. */
  template <class Line, class AllocCov>
  int extract(const float* data, int n_floats, std::vector<Line>& lines, AllocCov alloc_cov) {
    int n = 0;
    const int rc = ekf_lx_extract(lx_, n_floats / 2, data, &n, rows_.data());
    if (rc != EKF_OK) throw std::runtime_error(std::string("libekfcuda: ") + ekf_lx_last_error(lx_));
    if (n > max_lines_) n = max_lines_;
    for (int i = 0; i < n; ++i) {
      const double* o = &rows_[10 * (size_t)i];
      Line l;
      l.alfa = o[0]; l.r = o[1];
      l.C_AR = alloc_cov();
      for (int t = 0; t < 4; ++t) l.C_AR->data[t] = o[2 + t];
      for (int k = 0; k < 2; ++k) {
        typename decltype(l.lineInterval)::value_type p;
        p.alfa = o[6 + 2 * k]; p.r = o[7 + 2 * k];
        l.lineInterval.push_back(p);
      }
      lines.push_back(l);
    }
    return n;
  }

  /* lineprovider/main.cpp:60-84 (Transform) for the lines of the last extract(): appends 4 floats per line (x0, y0, x1, y1,
   * world frame) to `data` -- the `lines_1` message; scale = 100 gives the planner's centimetres (astar/main.cpp:44-73).
   * Returns the number of lines. */
  int worldSegments(double x, double y, double theta, std::vector<float>& data, double scale = 1.0) {
    const double pose[3] = {x, y, theta};
    std::vector<float> seg(4 * (size_t)max_lines_);
    int n = 0;
    const int rc = ekf_lx_world_segments(lx_, pose, scale, seg.data(), max_lines_, &n);
    if (rc != EKF_OK) throw std::runtime_error(std::string("libekfcuda: ") + ekf_lx_last_error(lx_));
    data.insert(data.end(), seg.begin(), seg.begin() + 4 * (size_t)n);
    return n;
  }

 private:
  ekf_lx* lx_;
  int max_lines_;
  std::vector<double> rows_;
};

}  // namespace ekfcuda
#endif
