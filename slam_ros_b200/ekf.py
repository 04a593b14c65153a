"""ctypes binding of libekfcuda.so (include/ekf.h).  Plumbing only: every call goes to the CUDA library.

Fails loudly when the library is missing or when no CUDA device is present -- there is no CPU path.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# EKF_LIB points diagnostics at an instrumented build of the same library (e.g. -DEKF_LINE_TIMING); default: in-tree
_LIB_PATH = os.environ.get("EKF_LIB") or os.path.join(_HERE, "libekfcuda.so")
_lib = None

EKF_OK, EKF_EINVAL, EKF_ECAPACITY, EKF_ESINGULAR, EKF_ECUDA, EKF_ENCCL, EKF_ENOMEM, EKF_ESTATE = range(8)
EKF_FLAG_EAGER_SWEEP = 1
EKF_FLAG_SWEEP_DIRECT = 2
EKF_FLAG_PER_LINE_KERNELS = 4
EKF_FLAG_NO_OVERLAP = 8
EKF_FLAG_FULL_GATES = 16
EKF_POSE_X, EKF_POSE_Y, EKF_POSE_THETA = 1, 2, 4
_STATUS = {0: "OK", 1: "EINVAL", 2: "ECAPACITY", 3: "ESINGULAR", 4: "ECUDA", 5: "ENCCL", 6: "ENOMEM", 7: "ESTATE"}

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_fp = C.POINTER(C.c_float)


class EkfConfig(C.Structure):
    _fields_ = [("capacity_lines", C.c_int), ("gate", C.c_double), ("encoder_noise", C.c_double),
                ("reset_headroom", C.c_int), ("device", C.c_int), ("max_batch", C.c_int), ("flags", C.c_int)]


class EkfError(RuntimeError):
    def __init__(self, code, where, detail=""):
        self.code = code
        super().__init__("%s -> %s%s" % (where, _STATUS.get(code, code), (": " + detail) if detail else ""))


def library_path():
    return _LIB_PATH


# every symbol include/ekf.h declares (tests check the .so exports exactly these)
SYMBOLS = [
    "ekf_default_config", "ekf_create", "ekf_destroy", "ekf_last_error", "ekf_predict", "ekf_associate",
    "ekf_update", "ekf_add_line", "ekf_end_scan", "ekf_scan", "ekf_scan_device", "ekf_sync", "ekf_get_state",
    "ekf_get_robot_cov", "ekf_get_ellipse", "ekf_download", "ekf_upload", "ekf_remove_lines", "ekf_insert_lines", "ekf_observe_pose",
    "ekf_download_live",
    "ekf_download_block", "ekf_cov_stats", "ekf_profile_enable", "ekf_profile_read", "ekf_profile_read_lines", "ekf_timer_start", "ekf_timer_stop", "ekf_sweep_probe",
    "ekf_nccl_unique_id", "ekf_create_sharded", "ekf_shard_ipc_handle", "ekf_shard_connect", "ekf_shard_use_fused", "ekf_batch_create", "ekf_batch_destroy", "ekf_batch_scan",
    "ekf_batch_submit", "ekf_batch_collect", "ekf_batch_scan_device", "ekf_batch_sync", "ekf_batch_download", "ekf_batch_last_error", "ekf_version",
    "ekf_lx_create", "ekf_lx_destroy", "ekf_lx_last_error", "ekf_lx_extract", "ekf_lx_extract_device", "ekf_lx_sync", "ekf_lx_world_segments",
]


def load_library():
    """dlopen libekfcuda.so.  Raises (never falls back) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise ImportError("libekfcuda.so is not built (%s). Run `python -m slam_ros_b200.build` "
                          "(needs nvcc); there is no CPU fallback." % _LIB_PATH)
    lib = C.CDLL(_LIB_PATH)
    vp = C.c_void_p
    lib.ekf_version.restype = C.c_char_p
    lib.ekf_last_error.restype = C.c_char_p
    lib.ekf_last_error.argtypes = [vp]
    lib.ekf_batch_last_error.restype = C.c_char_p
    lib.ekf_batch_last_error.argtypes = [vp]
    lib.ekf_default_config.argtypes = [C.POINTER(EkfConfig)]
    lib.ekf_create.argtypes = [C.POINTER(vp), C.POINTER(EkfConfig)]
    lib.ekf_create_sharded.argtypes = [C.POINTER(vp), C.POINTER(EkfConfig), C.c_int, C.c_int, C.c_char_p]
    lib.ekf_nccl_unique_id.argtypes = [C.c_char_p]
    lib.ekf_shard_ipc_handle.argtypes = [vp, C.c_char_p]
    lib.ekf_shard_connect.argtypes = [vp, C.c_char_p]
    lib.ekf_shard_use_fused.argtypes = [vp, C.c_int]
    lib.ekf_destroy.argtypes = [vp]
    lib.ekf_predict.argtypes = [vp, _dp, _dp, _dp]
    lib.ekf_associate.argtypes = [vp, _dp, _dp, _ip, _dp]
    lib.ekf_update.argtypes = [vp, C.c_int, _dp, _dp, _dp]
    lib.ekf_add_line.argtypes = [vp, _dp, _dp]
    lib.ekf_end_scan.argtypes = [vp, C.c_int, _dp]
    lib.ekf_scan.argtypes = [vp, _dp, _dp, C.c_int, _dp, _dp, _ip, _dp]
    lib.ekf_scan_device.argtypes = [vp, vp, C.c_int, vp, vp, vp]
    lib.ekf_sync.argtypes = [vp]
    lib.ekf_get_state.argtypes = [vp, _dp, _ip, _ip]
    lib.ekf_get_robot_cov.argtypes = [vp, _dp]
    lib.ekf_get_ellipse.argtypes = [vp, _fp, _fp, _ip]
    lib.ekf_download.argtypes = [vp, _dp, _dp, _ip]
    lib.ekf_upload.argtypes = [vp, _dp, _dp, C.c_int]
    lib.ekf_remove_lines.argtypes = [vp, C.c_int, _ip, _ip]
    lib.ekf_insert_lines.argtypes = [vp, C.c_int, _dp, _dp, _ip]
    lib.ekf_observe_pose.argtypes = [vp, C.c_int, _dp, _dp, C.c_double, _dp, _ip, _dp]
    lib.ekf_download_live.argtypes = [vp, _dp, _dp, C.c_int, C.c_int, _ip]
    lib.ekf_download_block.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, _dp]
    lib.ekf_cov_stats.argtypes = [vp, _dp, _dp, _dp]
    lib.ekf_profile_enable.argtypes = [vp, C.c_int]
    lib.ekf_profile_read.argtypes = [vp, _ip, _dp, _dp, C.POINTER(C.c_longlong)]
    lib.ekf_profile_read_lines.argtypes = [vp, _ip, _dp]
    lib.ekf_sweep_probe.argtypes = [vp, C.c_int, C.c_int, _dp]
    lib.ekf_timer_start.argtypes = [vp]
    lib.ekf_timer_stop.argtypes = [vp, _dp]
    lib.ekf_batch_create.argtypes = [C.POINTER(vp), C.POINTER(EkfConfig), C.c_int]
    lib.ekf_batch_destroy.argtypes = [vp]
    lib.ekf_batch_scan.argtypes = [vp, _dp, C.c_int, _dp, _dp, _ip, _dp]
    lib.ekf_batch_submit.argtypes = [vp, _dp, C.c_int, _dp, _dp]
    lib.ekf_batch_collect.argtypes = [vp, _ip, _dp]
    lib.ekf_batch_scan_device.argtypes = [vp, vp, C.c_int, vp, vp, vp]
    lib.ekf_batch_sync.argtypes = [vp]
    lib.ekf_batch_download.argtypes = [vp, C.c_int, _dp, _dp, _ip, _dp]
    lib.ekf_lx_create.argtypes = [C.POINTER(vp), C.c_int, C.c_int]
    lib.ekf_lx_destroy.argtypes = [vp]
    lib.ekf_lx_last_error.restype = C.c_char_p
    lib.ekf_lx_last_error.argtypes = [vp]
    lib.ekf_lx_extract.argtypes = [vp, C.c_int, C.POINTER(C.c_float), _ip, _dp]
    lib.ekf_lx_extract_device.argtypes = [vp, C.c_int, vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
    lib.ekf_lx_sync.argtypes = [vp]
    lib.ekf_lx_world_segments.argtypes = [vp, C.POINTER(C.c_double), C.c_double, C.POINTER(C.c_float), C.c_int, C.POINTER(C.c_int)]
    _lib = lib
    return lib


def _arr(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a


def _p(a):
    return a.ctypes.data_as(_dp) if a is not None else None


def default_config(**kw):
    lib = load_library()
    cfg = EkfConfig()
    lib.ekf_default_config(C.byref(cfg))
    for k, v in kw.items():
        if not hasattr(cfg, k):
            raise TypeError("unknown ekf_config field " + k)
        setattr(cfg, k, v)
    return cfg


class EkfFilter:
    """One ekf_ctx: a single filter whose state and covariance stay resident in HBM."""

    def __init__(self, capacity_lines=100, gate=0.4, encoder_noise=0.024, reset_headroom=10, device=0,
                 max_batch=64, flags=0, shard=None):
        """shard = (rank, world, nccl_unique_id_bytes) selects the row-sharded mode."""
        self._lib = load_library()
        self.cfg = default_config(capacity_lines=capacity_lines, gate=gate, encoder_noise=encoder_noise,
                                  reset_headroom=reset_headroom, device=device, max_batch=max_batch, flags=flags)
        self._h = C.c_void_p()
        if shard is None:
            rc = self._lib.ekf_create(C.byref(self._h), C.byref(self.cfg))
        else:
            rank, world, uid = shard
            rc = self._lib.ekf_create_sharded(C.byref(self._h), C.byref(self.cfg), int(rank), int(world), bytes(uid))
        if rc != EKF_OK:
            msg = self._lib.ekf_last_error(self._h).decode() if self._h else ""
            if self._h:
                self._lib.ekf_destroy(self._h)
                self._h = C.c_void_p()
            raise EkfError(rc, "ekf_create", msg)
        self.capacity = int(capacity_lines)
        self.n = 3 + 2 * self.capacity

    # -- plumbing ------------------------------------------------------------------------------
    def _check(self, rc, where, allow=()):
        if rc != EKF_OK and rc not in allow:
            raise EkfError(rc, where, self._lib.ekf_last_error(self._h).decode())
        return rc

    def close(self):
        if getattr(self, "_h", None):
            self._lib.ekf_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    # -- row-sharded mode: in-kernel NVLink exchange ------------------------------------------------
    def shard_ipc_handle(self):
        """64-byte CUDA IPC handle of this rank's exchange buffer."""
        buf = C.create_string_buffer(64)
        self._check(self._lib.ekf_shard_ipc_handle(self._h, buf), "ekf_shard_ipc_handle")
        return buf.raw

    def shard_connect(self, handles):
        """handles: the ranks' IPC handles in rank order (list of 64-byte strings).  Returns True when the peers
        are mapped; the fused exchange is switched on by shard_use_fused once ALL ranks report True."""
        blob = b"".join(bytes(h) for h in handles)
        rc = self._lib.ekf_shard_connect(self._h, blob)
        if rc == EKF_ECUDA:
            return False
        self._check(rc, "ekf_shard_connect")
        return True

    def shard_use_fused(self, on=True):
        """Every rank must make the same choice (parallel.connect_shards does the agreement)."""
        self._check(self._lib.ekf_shard_use_fused(self._h, 1 if on else 0), "ekf_shard_use_fused")

    # -- step-wise path (one call per reference block) -----------------------------------------------
    def predict(self, u, x_t0=None):
        ua = _arr(u, (3,)); xa = _arr(x_t0, (3,)) if x_t0 is not None else None
        out = np.zeros(3)
        self._check(self._lib.ekf_predict(self._h, _p(xa), _p(ua), _p(out)), "ekf_predict")
        return out

    def associate(self, z, R):
        za = _arr(z, (2,)); Ra = _arr(R, (4,)); j = C.c_int(-1); innov = np.zeros(2)
        self._check(self._lib.ekf_associate(self._h, _p(za), _p(Ra), C.byref(j), _p(innov)), "ekf_associate")
        return int(j.value), innov

    def update(self, j, z, R):
        za = _arr(z, (2,)); Ra = _arr(R, (4,)); out = np.zeros(3)
        self._check(self._lib.ekf_update(self._h, int(j), _p(za), _p(Ra), _p(out)), "ekf_update")
        return out

    def add_line(self, z, R):
        za = _arr(z, (2,)); Ra = _arr(R, (4,))
        self._check(self._lib.ekf_add_line(self._h, _p(za), _p(Ra)), "ekf_add_line")

    def end_scan(self, n_lines):
        pose = np.zeros(3)
        rc = self._check(self._lib.ekf_end_scan(self._h, int(n_lines), _p(pose)), "ekf_end_scan",
                         allow=(EKF_ECAPACITY, EKF_ESINGULAR))
        return rc, pose

    # -- fused path ------------------------------------------------------------------------------
    def scan(self, u, z, R, x_t0=None):
        """One whole Robot::localize.  Returns (status, j_out, pose)."""
        ua = _arr(u, (3,)); xa = _arr(x_t0, (3,)) if x_t0 is not None else None
        za = _arr(z).reshape(-1, 2); Ra = _arr(R).reshape(-1, 4)
        m = za.shape[0]
        j = np.full(max(m, 1), -1, dtype=np.int32); pose = np.zeros(3)
        rc = self._check(self._lib.ekf_scan(self._h, _p(xa), _p(ua), m, _p(za) if m else None, _p(Ra) if m else None,
                                            j.ctypes.data_as(_ip), _p(pose)), "ekf_scan",
                         allow=(EKF_ECAPACITY, EKF_ESINGULAR))
        return rc, j[:m], pose

    def scan_device(self, d_u, m, d_z, d_R, d_j_out=0):
        """Asynchronous scan on device-resident inputs (raw device addresses, e.g. tensor.data_ptr())."""
        self._check(self._lib.ekf_scan_device(self._h, C.c_void_p(d_u), int(m), C.c_void_p(d_z), C.c_void_p(d_R),
                                              C.c_void_p(d_j_out) if d_j_out else None), "ekf_scan_device")

    def sync(self):
        self._check(self._lib.ekf_sync(self._h), "ekf_sync")

    # -- state access ----------------------------------------------------------------------------
    def state(self):
        pose = np.zeros(3); L = C.c_int(0); st = C.c_int(0)
        self._check(self._lib.ekf_get_state(self._h, _p(pose), C.byref(L), C.byref(st)), "ekf_get_state")
        return pose, int(L.value), int(st.value)

    @property
    def lines(self):
        return self.state()[1]

    @property
    def pose(self):
        return self.state()[0]

    def robot_cov(self):
        out = np.zeros(9)
        self._check(self._lib.ekf_get_robot_cov(self._h, _p(out)), "ekf_get_robot_cov")
        return out.reshape(3, 3)

    def get_ellipse(self):
        ax = (C.c_float * 2)(); ang = C.c_float(0); ok = C.c_int(0)
        self._check(self._lib.ekf_get_ellipse(self._h, ax, C.byref(ang), C.byref(ok)), "ekf_get_ellipse")
        return bool(ok.value), (float(ax[0]), float(ax[1])), float(ang.value)

    def download(self):
        """(y[n], P[n,n], n_lines) in the reference's capacity layout."""
        y = np.zeros(self.n); P = np.zeros((self.n, self.n)); L = C.c_int(0)
        self._check(self._lib.ekf_download(self._h, _p(y), _p(P), C.byref(L)), "ekf_download")
        return y, P, int(L.value)

    def download_live(self):
        L = self.lines
        nl = 3 + 2 * L
        y = np.zeros(nl); P = np.zeros((nl, nl)); Lc = C.c_int(0)
        self._check(self._lib.ekf_download_live(self._h, _p(y), _p(P), nl, nl, C.byref(Lc)), "ekf_download_live")
        return y, P, int(Lc.value)

    def download_y(self):
        L = self.lines
        nl = 3 + 2 * L
        y = np.zeros(nl); Lc = C.c_int(0)
        self._check(self._lib.ekf_download_live(self._h, _p(y), None, nl, nl, C.byref(Lc)), "ekf_download_live")
        return y

    def download_block(self, r0, c0, nr, nc):
        out = np.zeros((nr, nc))
        self._check(self._lib.ekf_download_block(self._h, int(r0), int(c0), int(nr), int(nc), _p(out)), "ekf_download_block")
        return out

    def upload(self, y, P, n_lines):
        ya = _arr(y, (self.n,)); Pa = _arr(P, (self.n, self.n))
        self._check(self._lib.ekf_upload(self._h, _p(ya), _p(Pa), int(n_lines)), "ekf_upload")

    def remove_lines(self, indices):
        """Removes landmarks `indices` (strictly increasing, each below the line count) from the map: their entries of y
        and rows and columns of P go, later landmarks move down in order.  Returns the new line count."""
        idx = np.ascontiguousarray(np.asarray(indices, dtype=np.int32).reshape(-1))
        L = C.c_int(0)
        self._check(self._lib.ekf_remove_lines(self._h, idx.size, idx.ctypes.data_as(_ip) if idx.size else None,
                                               C.byref(L)), "ekf_remove_lines")
        return int(L.value)

    def insert_lines(self, lines, cov=None):
        """Appends k known landmarks after the existing ones: lines = k x (alfa, r) in the world frame (alfa wrapped as
        the augmentation wraps it), cov = None (surveyed: zero covariance, fixed from then on) or their 2k x 2k joint
        covariance; zero cross-covariance with the rest.  All or nothing (EKF_ECAPACITY when they do not fit).  Returns
        the new line count."""
        la = _arr(lines).reshape(-1)
        if la.size % 2:
            raise ValueError("insert_lines: lines must be (alfa, r) pairs")
        k = la.size // 2
        ca = _arr(cov, (2 * k, 2 * k)) if cov is not None else None
        L = C.c_int(0)
        self._check(self._lib.ekf_insert_lines(self._h, k, _p(la) if k else None, _p(ca), C.byref(L)), "ekf_insert_lines")
        return int(L.value)

    def observe_pose(self, z, R, mask=7, d2_max=float("inf")):
        """Fuses an absolute measurement of the components `mask` selects (EKF_POSE_X | EKF_POSE_Y | EKF_POSE_THETA) of
        the pose: z = (x, y, theta), R = its 3x3 covariance (only the selected entries are read).  The fix is accepted
        iff S is nonsingular and d2 <= d2_max.  Returns (status, accepted, d2, pose): status EKF_OK, or EKF_ESINGULAR for
        a singular S (state unchanged); pose = the resulting xPos, yPos, thetaPos."""
        za = _arr(z, (3,)); Ra = _arr(R, (9,)); d2 = C.c_double(0); acc = C.c_int(0); pose = np.zeros(3)
        rc = self._check(self._lib.ekf_observe_pose(self._h, int(mask), _p(za), _p(Ra), float(d2_max), C.byref(d2),
                                                    C.byref(acc), _p(pose)), "ekf_observe_pose", allow=(EKF_ESINGULAR,))
        return rc, bool(acc.value), float(d2.value), pose

    def cov_stats(self):
        t = C.c_double(0); s = C.c_double(0); q = C.c_double(0)
        self._check(self._lib.ekf_cov_stats(self._h, C.byref(t), C.byref(s), C.byref(q)), "ekf_cov_stats")
        return t.value, s.value, q.value

    # -- measurement -----------------------------------------------------------------------------
    def profile_enable(self, on=True):
        self._check(self._lib.ekf_profile_enable(self._h, 1 if on else 0), "ekf_profile_enable")

    def profile_read(self):
        ns = C.c_int(0); ms = C.c_double(0); by = C.c_double(0); ln = C.c_longlong(0)
        self._check(self._lib.ekf_profile_read(self._h, C.byref(ns), C.byref(ms), C.byref(by), C.byref(ln)), "ekf_profile_read")
        return {"sweeps": int(ns.value), "sweep_ms": ms.value, "sweep_bytes": by.value, "launches": int(ln.value)}

    def profile_read_lines(self):
        ns = C.c_int(0); ms = C.c_double(0)
        self._check(self._lib.ekf_profile_read_lines(self._h, C.byref(ns), C.byref(ms)), "ekf_profile_read_lines")
        return {"scans": int(ns.value), "line_ms": ms.value}

    def timer_start(self):
        self._check(self._lib.ekf_timer_start(self._h), "ekf_timer_start")

    def timer_stop(self):
        ms = C.c_double(0)
        self._check(self._lib.ekf_timer_stop(self._h, C.byref(ms)), "ekf_timer_stop")
        return ms.value

    def sweep_probe(self, m=1, repeats=10):
        ms = C.c_double(0)
        self._check(self._lib.ekf_sweep_probe(self._h, int(m), int(repeats), C.byref(ms)), "ekf_sweep_probe")
        return ms.value


def nccl_unique_id():
    lib = load_library()
    buf = C.create_string_buffer(128)
    rc = lib.ekf_nccl_unique_id(buf)
    if rc != EKF_OK:
        raise EkfError(rc, "ekf_nccl_unique_id", "libnccl.so.2 not loadable")
    return buf.raw


class EkfBatch:
    """B independent filters on one device (Monte-Carlo batch); one thread block per filter."""

    def __init__(self, n_filters, capacity_lines=50, gate=0.4, encoder_noise=0.024, reset_headroom=10, device=0, flags=0):
        self._lib = load_library()
        self.cfg = default_config(capacity_lines=capacity_lines, gate=gate, encoder_noise=encoder_noise,
                                  reset_headroom=reset_headroom, device=device, flags=flags)
        self._h = C.c_void_p()
        rc = self._lib.ekf_batch_create(C.byref(self._h), C.byref(self.cfg), int(n_filters))
        if rc != EKF_OK:
            msg = self._lib.ekf_batch_last_error(self._h).decode() if self._h else ""
            if self._h:
                self._lib.ekf_batch_destroy(self._h)
                self._h = C.c_void_p()
            raise EkfError(rc, "ekf_batch_create", msg)
        self.B = int(n_filters)
        self.capacity = int(capacity_lines)
        self.n = 3 + 2 * self.capacity
        self._pending = []           # line counts of the submitted, not yet collected steps

    def _check(self, rc, where, allow=()):
        if rc != EKF_OK and rc not in allow:
            raise EkfError(rc, where, self._lib.ekf_batch_last_error(self._h).decode())
        return rc

    def _lines(self, u, z, R):
        """u (B,3), z (B,m,2), R (B,m,4) as contiguous doubles; m may be 0."""
        za = _arr(z); Ra = _arr(R)
        m = za.size // (2 * self.B)
        return _arr(u, (self.B, 3)), za.reshape(self.B, m, 2), Ra.reshape(self.B, m, 4), m
        return rc

    def close(self):
        if getattr(self, "_h", None):
            self._lib.ekf_batch_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def scan(self, u, z, R):
        """u (B,3), z (B,m,2), R (B,m,4) -> (status, j_out (B,m), pose (B,3))."""
        ua, za, Ra, m = self._lines(u, z, R)
        j = np.full((self.B, max(m, 1)), -1, dtype=np.int32); pose = np.zeros((self.B, 3))
        rc = self._check(self._lib.ekf_batch_scan(self._h, _p(ua), m, _p(za) if m else None, _p(Ra) if m else None,
                                                  j.ctypes.data_as(_ip), _p(pose)), "ekf_batch_scan",
                         allow=(EKF_ECAPACITY, EKF_ESINGULAR))
        return rc, j[:, :m], pose

    def submit(self, u, z, R):
        """Pipelined host path: stage one step and return at once (at most two in flight); results come from collect()."""
        ua, za, Ra, m = self._lines(u, z, R)
        self._check(self._lib.ekf_batch_submit(self._h, _p(ua), m, _p(za) if m else None, _p(Ra) if m else None), "ekf_batch_submit")
        self._pending.append(m)

    def collect(self):
        """(status, j_out (B,m), pose (B,3)) of the OLDEST submitted step."""
        m = self._pending[0] if self._pending else 0
        j = np.full((self.B, max(m, 1)), -1, dtype=np.int32); pose = np.zeros((self.B, 3))
        rc = self._check(self._lib.ekf_batch_collect(self._h, j.ctypes.data_as(_ip), _p(pose)), "ekf_batch_collect",
                         allow=(EKF_ECAPACITY, EKF_ESINGULAR))
        self._pending.pop(0)
        return rc, j[:, :m], pose

    def scan_device(self, d_u, m, d_z, d_R, d_j_out=0):
        self._check(self._lib.ekf_batch_scan_device(self._h, C.c_void_p(d_u), int(m), C.c_void_p(d_z), C.c_void_p(d_R),
                                                    C.c_void_p(d_j_out) if d_j_out else None), "ekf_batch_scan_device")

    def sync(self):
        self._check(self._lib.ekf_batch_sync(self._h), "ekf_batch_sync")

    def download(self, f):
        y = np.zeros(self.n); P = np.zeros((self.n, self.n)); L = C.c_int(0); pose = np.zeros(3)
        self._check(self._lib.ekf_batch_download(self._h, int(f), _p(y), _p(P), C.byref(L), _p(pose)), "ekf_batch_download")
        return y, P, int(L.value), pose


class LineExtractor:
    """ekf_lx: the node's `mapping_cb` + LineExtraction (slam_ros/main.cpp:37-71, lineFitting.cpp:640-702) on the
    device.  extract(payload) -> (rows, n): rows[i] = alfa, r, C_AR[4], interval0 (alfa, r), interval1 (alfa, r)."""

    def __init__(self, device=0, max_lines=128):
        self._lib = load_library()
        self._h = C.c_void_p()
        self.max_lines = int(max_lines)
        rc = self._lib.ekf_lx_create(C.byref(self._h), int(device), self.max_lines)
        if rc != EKF_OK:
            msg = self._lib.ekf_lx_last_error(self._h).decode() if self._h else ""
            if self._h:
                self._lib.ekf_lx_destroy(self._h)
                self._h = C.c_void_p()
            raise EkfError(rc, "ekf_lx_create", msg)

    def _check(self, rc, where):
        if rc != EKF_OK:
            raise EkfError(rc, where, self._lib.ekf_lx_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None):
            self._lib.ekf_lx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def extract(self, payload):
        d = np.ascontiguousarray(np.asarray(payload, dtype=np.float32).reshape(-1))
        out = np.zeros((self.max_lines, 10)); n = C.c_int(0)
        self._check(self._lib.ekf_lx_extract(self._h, d.size // 2, d.ctypes.data_as(C.POINTER(C.c_float)), C.byref(n),
                                             _p(out)), "ekf_lx_extract")
        return out[:min(n.value, self.max_lines)].copy(), int(n.value)

    def extract_device(self, d_payload, n_pairs):
        """Payload already in HBM (raw device address).  Returns the device addresses (z, R, count) of the result."""
        z = C.c_void_p(); R = C.c_void_p(); cnt = C.c_void_p()
        self._check(self._lib.ekf_lx_extract_device(self._h, int(n_pairs), C.c_void_p(d_payload), C.byref(z), C.byref(R),
                                                    C.byref(cnt)), "ekf_lx_extract_device")
        return z.value, R.value, cnt.value

    def world_segments(self, pose, scale=1.0):
        """lineprovider's Transform (main.cpp:60-84) on the lines of the last extraction: (n, 4) float32 world-frame end
        points (x0, y0, x1, y1), i.e. the `lines_1` message; scale=100: the planner's centimetres (astar/main.cpp:44-73)."""
        ps = np.ascontiguousarray(np.asarray(pose, dtype=np.float64).reshape(3))
        out = np.zeros((self.max_lines, 4), dtype=np.float32); n = C.c_int(0)
        self._check(self._lib.ekf_lx_world_segments(self._h, _p(ps), float(scale), out.ctypes.data_as(C.POINTER(C.c_float)),
                                                    self.max_lines, C.byref(n)), "ekf_lx_world_segments")
        return out[:min(n.value, self.max_lines)].copy()

    def sync(self):
        self._check(self._lib.ekf_lx_sync(self._h), "ekf_lx_sync")
