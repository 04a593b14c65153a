"""Host-side mirror of the reference's `Robot` class (slam_ros/Robot.h:21-77) over libekfcuda.

Same public names and argument meaning as the reference so that parity tests read like calls into the
reference: ``Robot(x, y, theta)``, ``localize(lines, rot, encoder)``, ``getEllipse()``, the pose mirrors
``xPos / yPos / thetaPos``, ``P_t0`` and ``lineIntervals``.  All arithmetic of the filter runs on the GPU;
the only host arithmetic is what the reference also does outside GSL: the odometry vector built from
(pose - encoder) (Robot.cpp:135-145) and the float endpoints of new lines (Robot.cpp:869-879).

The C++ equivalent a slam_ros maintainer would compile into the node is include/ekf_robot.hpp.
"""
import math
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

import numpy as np

from .ekf import EkfFilter, EKF_OK

LINESIZE = 100          # Robot.h:13
MAHALANOBIS = 0.4       # Robot.h:15
ENCODERNOISE = 0.024    # Robot.h:17
SIMULATIONOFF = True    # Robot.h:18


@dataclass
class Line:
    """simplifyPath.h:62-79: `alfa` first, then `r`; C_AR is the 2x2 covariance of (alfa, r), row-major;
    lineInterval holds 0 or 2 end points as (alfa, r) polar pairs in the robot frame."""
    alfa: float
    r: float
    C_AR: Sequence[float] = (0.0, 0.0, 0.0, 0.0)
    lineInterval: List[Tuple[float, float]] = field(default_factory=list)


def _libm_float_trig():
    """cosf / sinf of the C library: `cos(alpha)` with `float alpha` inside Robot.cpp resolves to std::cos(float)
    (<cmath> + `using namespace std`, simplifyPath.h:16-24), and numpy's float32 kernels round differently."""
    import ctypes
    import ctypes.util
    try:
        lm = ctypes.CDLL(ctypes.util.find_library("m") or "libm.so.6")
        lm.cosf.restype = ctypes.c_float; lm.cosf.argtypes = [ctypes.c_float]
        lm.sinf.restype = ctypes.c_float; lm.sinf.argtypes = [ctypes.c_float]
        return lm.cosf, lm.sinf
    except Exception:                                     # no C library to ask: numpy's float32 kernels (<= 1 ulp apart)
        return (lambda a: float(np.cos(np.float32(a)))), (lambda a: float(np.sin(np.float32(a))))


_cosf, _sinf = _libm_float_trig()


def interval_end_point(alpha, r, x, y, theta):
    """One end point of an appended line as the node publishes it on `lines` (Robot.cpp:870-873), two float32 values:
    `float alpha` (:871); cos / sin of that float are the FLOAT functions; polar_point(alfa, r) scales its first
    argument by PI/180 with PI = 3.14159265 (lineFitting.cpp:71-77, lineFitting.h:12) -- reproduced, it is what the
    node publishes; polar2descart (lineFitting.cpp:170-176); the result is pushed into a std::vector<float>.
    Checked float for float against the reference itself (tests/test_oracle.py: 5304 values, 0 differ)."""
    alpha = float(np.float32(alpha))
    rad = r + x * float(_cosf(alpha)) + y * float(_sinf(alpha))
    a = (alpha + theta) * (3.14159265 / 180)
    return float(np.float32(math.cos(a) * rad)), float(np.float32(math.sin(a) * rad))


class Robot:
    def __init__(self, x=0.0, y=0.0, theta=0.0, linesize=LINESIZE, device=0, **cfg):
        self._f = EkfFilter(capacity_lines=linesize, gate=cfg.pop("gate", MAHALANOBIS),
                            encoder_noise=cfg.pop("encoder_noise", ENCODERNOISE), device=device, **cfg)
        self.xPos, self.yPos, self.thetaPos = float(x), float(y), float(theta)     # Robot.cpp:22-24
        self.lineIntervals: List[float] = []                                          # Robot.h:59 (float32 data)
        self.last_matches: Optional[np.ndarray] = None
        self.last_status = EKF_OK

    @property
    def filter(self):
        return self._f

    @property
    def savedLineCount(self):
        return self._f.lines

    @property
    def P_t0(self):
        """Robot.h:62: SLAMSIZE x SLAMSIZE row-major covariance (downloaded, symmetrised)."""
        return self._f.download()[1]

    @property
    def y(self):
        return self._f.download()[0]

    def localize(self, lines: Sequence[Line], rot=None, encoder=None):
        """Robot::localize (Robot.cpp:126-943).  `rot` is accepted for signature parity and ignored, as in
        the reference when SIMULATIONOFF is true (Robot.cpp:136-145); `encoder` is the external pose."""
        if encoder is None:
            raise ValueError("encoder pose is required (the reference dereferences it when SIMULATIONOFF)")
        x_t0 = (self.xPos, self.yPos, self.thetaPos)                                  # Robot.cpp:130
        dX, dY = x_t0[0] - encoder[0], x_t0[1] - encoder[1]
        u = (math.sqrt(dX * dX + dY * dY), 0.0, x_t0[2] - encoder[2])                 # Robot.cpp:141-144 (Q5)
        m = len(lines)
        z = np.array([[ln.alfa, ln.r] for ln in lines], dtype=np.float64).reshape(m, 2)
        R = np.array([list(ln.C_AR) for ln in lines], dtype=np.float64).reshape(m, 4)
        L_before = self._f.lines
        rc, j, pose = self._f.scan(u, z, R, x_t0=x_t0)
        self.last_status, self.last_matches = rc, j
        self.xPos, self.yPos, self.thetaPos = float(pose[0]), float(pose[1]), float(pose[2])
        # STORING LINE INTERVALS (Robot.cpp:869-879): end points of every line that was appended
        room = max(0, self._f.capacity - L_before)
        added = 0
        for i, ln in enumerate(lines):
            if j[i] >= 0:
                continue
            if added >= room:
                break
            added += 1
            if len(ln.lineInterval) == 2:
                for (alpha, rr) in (ln.lineInterval[0], ln.lineInterval[-1]):
                    self.lineIntervals.extend(interval_end_point(alpha, rr, self.xPos, self.yPos, self.thetaPos))
        return rc

    def remove_lines(self, indices):
        """Not in the reference: removes landmarks `indices` (strictly increasing) from the map (ekf_remove_lines).
        savedLineCount follows; lineIntervals, the per-scan log the node clears after publishing, is untouched.
        Returns the new savedLineCount."""
        return self._f.remove_lines(indices)

    def observe_pose(self, z, R, mask=7, d2_max=float("inf")):
        """Not in the reference: fuses an absolute pose measurement (ekf_observe_pose; z = (x, y, theta), R its 3x3
        covariance, mask of EKF_POSE_X | EKF_POSE_Y | EKF_POSE_THETA).  The pose mirrors xPos / yPos / thetaPos follow
        the corrected pose: `localize` passes them as x_t0 (Robot.cpp:130), so a stale mirror would overwrite the fix at
        the next prediction.  As after any update, the next `localize` forms its odometry from the corrected pose and
        the encoder pose (Robot.cpp:140-145, SURVEY Q5).  Returns (status, accepted, d2)."""
        rc, acc, d2, pose = self._f.observe_pose(z, R, mask=mask, d2_max=d2_max)
        self.xPos, self.yPos, self.thetaPos = float(pose[0]), float(pose[1]), float(pose[2])
        return rc, acc, d2

    def getEllipse(self):
        """Robot::getEllipse (Robot.cpp:73-124) -> (ok, (axis0, axis1), angle)."""
        return self._f.get_ellipse()

    def robotPosition(self):
        """The node's `robotPosition` message (slam_ros/main.cpp:150-169): translation (x, y, theta) and
        rotation.x/.y/.z = major axis, minor axis, ellipse angle."""
        ok, ax, ang = self.getEllipse()
        return {"translation": (self.xPos, self.yPos, self.thetaPos), "rotation": (ax[1], ax[0], ang), "ellipse_ok": ok}
