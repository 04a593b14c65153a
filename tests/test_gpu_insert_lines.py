"""ekf_insert_lines: known landmarks appended to a resident map (y' = [y, lines], P' = [[P, 0], [0, C]]).

1. Bitwise against numpy on the downloaded state, on the out-of-place path (second covariance buffer) and the in-place
   path (EKF_FLAG_NO_OVERLAP), which must also agree with each other, at 3 300 and 12 000 landmarks and on an empty map.
2. Insert == upload: two filters run the same scans; at the same point one inserts and the other uploads the numpy-built
   state; afterwards associations, y and P stay identical bit for bit, whatever the pipeline held at the insertion.
3. Surveyed landmarks (zero covariance) stay fixed under every scan path: their y entries do not change and their rows
   of P stay zero, while every scan matches them.
4. Against the structured CPU oracle: a floor plan (the room's walls) inserted on a fresh filter, and a prior block
   inserted in the middle of a 3 300-landmark run.
5. Componentwise against the extended-precision reference after an insertion with a prior covariance.
6. Errors leave the state bitwise unchanged.
7. The Python and C++ mirrors (Robot.insert_lines, Robot::insertLines).
"""
import ctypes as C
import math
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import hp_reference as hp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TESTS = os.path.dirname(os.path.abspath(__file__))
OVERLAP_MIN_N = 6000        # kOverlapMinN (ekf_api.cu): below this state dimension scans do not overlap
U = (0.02, 0.0, 0.01)


def wrap(a):
    """normalize_radian (Robot.cpp:62-71) in float64, operation for operation as the device evaluates it."""
    a = float(a)
    if a > math.pi:
        return a - (2.0 * math.pi + (math.floor(a / (2.0 * math.pi)) * 2.0) * math.pi)
    if a < -math.pi:
        return a + (2.0 * math.pi + (math.floor(abs(a) / (2.0 * math.pi)) * 2.0) * math.pi)
    return a


def np_insert(y0, P0, lines, cov):
    """The expected live state after the insertion."""
    ln = np.array(lines, dtype=np.float64).reshape(-1, 2)
    ln[:, 0] = [wrap(a) for a in ln[:, 0]]
    nl0, k = y0.size, ln.shape[0]
    y = np.concatenate([y0, ln.ravel()])
    P = np.zeros((nl0 + 2 * k, nl0 + 2 * k))
    P[:nl0, :nl0] = P0
    if cov is not None:
        P[nl0:, nl0:] = cov
    return y, P


def layout(y, P, n):
    """A live state in the capacity layout ekf_upload takes."""
    Y = np.zeros(n); Y[:y.size] = y
    PP = np.zeros((n, n)); PP[:y.size, :y.size] = P
    return Y, PP


def spd(k, rng, scale=1e-4):
    """An exactly symmetric positive definite 2k x 2k covariance."""
    A = rng.standard_normal((2 * k, 2 * k + 3))
    M = (A @ A.T / (2 * k + 3) + 0.1 * np.eye(2 * k)) * scale
    return np.triu(M) + np.triu(M, 1).T


def random_lines(k, rng, r=(1.0, 9.0)):
    return np.stack([rng.uniform(-math.pi, math.pi, k), rng.uniform(r[0], r[1], k)], axis=1)


def seeded_map(N, cap, steps, flags=0, seed=11, **kw):
    from slam_ros_b200 import EkfFilter, scenario as sc
    scn = sc.map_scenario(N, steps, m=8, seed=seed)
    f = EkfFilter(capacity_lines=cap, flags=flags, **kw)
    f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    for s in range(steps):
        f.scan(scn["u"][s], scn["z"][s], scn["R"][s])
    return f


# ---- 1. bitwise against numpy ---------------------------------------------------------------------------------------
def test_insert_lines_bitwise_against_numpy_3300(libekf):
    """3 300 landmarks (overlapped path, n >= 6000), capacity 3 400: every case on a fresh copy of the same state, on
    both paths.  nl = 6 603 = 11 (mod 64), so blocks of 26 and 27 landmarks end at nl' = 63 and 1 (mod 64), and every
    block of 27 or more straddles the tile edge at 6 656."""
    from slam_ros_b200.ekf import EKF_FLAG_NO_OVERLAP
    N, cap = 3300, 3400
    fs = {"oop": seeded_map(N, cap, 5), "inplace": seeded_map(N, cap, 5, flags=EKF_FLAG_NO_OVERLAP)}
    y0, P0, L0 = fs["oop"].download_live()
    assert L0 == fs["inplace"].lines == N and 3 + 2 * L0 >= OVERLAP_MIN_N
    Y, P = layout(y0, P0, 3 + 2 * cap)
    rng = np.random.default_rng(3)
    nl0 = y0.size
    k1, k63 = ((1 - nl0) % 64) // 2, ((63 - nl0) % 64) // 2
    cases = [("surveyed_k1", 1, False), ("spd_k1", 1, True), ("spd_k37", 37, True), ("nl1", k1, True),
             ("nl63", k63, False), ("tile_edge", 30, True), ("to_capacity", cap - N, True),
             ("to_capacity_surveyed", cap - N, False)]
    for name, k, with_cov in cases:
        lines = random_lines(k, rng)
        cov = spd(k, rng) if with_cov else None
        ye, Pe = np_insert(y0, P0, lines, cov)
        if name in ("nl1", "nl63"):
            assert ye.size % 64 == int(name[2:])
        got = {}
        for path, f in fs.items():
            f.upload(Y, P, L0)
            pose0, rcov0 = f.pose, f.robot_cov()
            Ln = f.insert_lines(lines, cov)
            y, Pn, L = f.download_live()
            assert Ln == L == L0 + k, (name, path)
            assert np.array_equal(y, ye), (name, path)
            assert np.array_equal(Pn, Pe), (name, path, np.argwhere(Pn != Pe)[:5])
            assert np.array_equal(f.pose, pose0) and np.array_equal(f.robot_cov(), rcov0), (name, path)
            got[path] = (y, Pn)
        assert all(np.array_equal(a, b) for a, b in zip(got["oop"], got["inplace"])), name
    for f in fs.values():
        f.close()


def test_insert_lines_bitwise_on_an_empty_map(libekf):
    """An empty filter filled to capacity in one call, with and without a covariance, on both paths; angles outside
    (-pi, pi] are wrapped as the augmentation wraps them; k = 0 is a no-op."""
    from slam_ros_b200 import EkfFilter
    from slam_ros_b200.ekf import EKF_FLAG_NO_OVERLAP
    rng = np.random.default_rng(7)
    cap = 40
    lines = random_lines(cap, rng)
    lines[:6, 0] = [4.0, -7.5, 3.0 * math.pi, math.pi, -math.pi, 40.0]
    for flags in (0, EKF_FLAG_NO_OVERLAP):
        for cov in (None, spd(cap, rng)):
            f = EkfFilter(capacity_lines=cap, flags=flags)
            y0, P0, L0 = f.download_live()
            assert L0 == 0
            assert f.insert_lines(np.zeros((0, 2))) == 0
            assert f.insert_lines(lines, cov) == cap
            ye, Pe = np_insert(y0, P0, lines, cov)
            y, P, L = f.download_live()
            assert L == cap and np.array_equal(y, ye) and np.array_equal(P, Pe), (flags, cov is None)
            assert abs(y[3]) <= math.pi and y[3] != 4.0
            assert f.insert_lines([]) == cap
            f.close()


def test_insert_lines_bitwise_against_numpy_12000(libekf):
    """12 000 landmarks, capacity 12 100: y, the robot rows and a set of 64 x 64 blocks (those around the new block
    included), each against the same block before the insertion (zero outside the old live part) plus the new block."""
    from slam_ros_b200.ekf import EKF_FLAG_NO_OVERLAP
    N, cap, k = 12000, 12100, 40
    fs = {"oop": seeded_map(N, cap, 3), "inplace": seeded_map(N, cap, 3, flags=EKF_FLAG_NO_OVERLAP)}
    rng = np.random.default_rng(5)
    lines = random_lines(k, rng)
    cov = spd(k, rng)
    nl0 = 3 + 2 * N
    nl = nl0 + 2 * k
    e = 64 * (nl0 // 64)
    edges = sorted({0, 128, 192 - 32, e - 64, e, nl - 64} | {int(v) * 64 for v in rng.integers(0, nl // 64, 10)})
    spots = [(r, c) for r in edges for c in edges if r <= c and r < nl and c < nl]
    got = {}
    for path, f in fs.items():
        y_old = f.download_y()
        top_old = f.download_block(0, 0, 3, nl0)
        pose0, rcov0 = f.pose, f.robot_cov()
        exp = []
        for r0, c0 in spots:
            nr, nc = min(64, nl - r0), min(64, nl - c0)
            B = f.download_block(r0, c0, nr, nc)
            for i in range(nr):
                if r0 + i >= nl0:
                    cs = max(c0, nl0)
                    B[i, cs - c0:] = cov[r0 + i - nl0, cs - nl0:c0 + nc - nl0]
            exp.append(B)
        assert f.insert_lines(lines, cov) == f.lines == N + k
        y = f.download_y()
        assert np.array_equal(y, np_insert(y_old, np.zeros((nl0, nl0)), lines, None)[0]), path
        top = f.download_block(0, 0, 3, nl)
        assert np.array_equal(top[:, :nl0], top_old) and not top[:, nl0:].any(), path
        blocks = [f.download_block(r0, c0, min(64, nl - r0), min(64, nl - c0)) for r0, c0 in spots]
        for (r0, c0), B, E in zip(spots, blocks, exp):
            assert np.array_equal(B, E), (path, r0, c0)
        assert np.array_equal(f.pose, pose0) and np.array_equal(f.robot_cov(), rcov0), path
        got[path] = [y, top] + blocks
    assert all(np.array_equal(a, b) for a, b in zip(got["oop"], got["inplace"]))
    for f in fs.values():
        f.close()


# ---- 2. insert == upload --------------------------------------------------------------------------------------------
class Twins:
    """Two filters fed the same scans; `insert` inserts on the first and uploads the numpy-built state on the second.
    ekf_upload sets the pose from y[0:3] while a scan leaves theta wrapped in the pose only, so the first scan after an
    insertion passes the pose from before it as x_t0 to both."""

    def __init__(self, N, cap, seed, max_batch=64, flags=0, m=8, S=220):
        from slam_ros_b200 import scenario as sc
        self.scn = sc.map_scenario(N, S, m=m, seed=seed)
        self.f = seeded_map(N, cap, 0, flags=flags, seed=seed, max_batch=max_batch)
        self.g = seeded_map(N, cap, 0, flags=flags, seed=seed, max_batch=max_batch)
        self.x_t0 = None
        self.J = []

    def scan(self, s, z=None, R=None):
        u = self.scn["u"][s]
        z = self.scn["z"][s] if z is None else z
        R = self.scn["R"][s] if R is None else R
        a = self.f.scan(u, z, R, x_t0=self.x_t0)
        b = self.g.scan(u, z, R, x_t0=self.x_t0)
        self.x_t0 = None
        assert np.array_equal(a[1], b[1]) and a[0] == b[0] and np.array_equal(a[2], b[2]), s
        self.J.append(a[1])
        return a[1]

    def stepwise(self, s):
        u, z, R = self.scn["u"][s], self.scn["z"][s], self.scn["R"][s]
        outs = []
        for f in (self.f, self.g):
            f.predict(u, x_t0=self.x_t0)
            j = np.full(len(z), -1, np.int32)
            for i in range(len(z)):
                j[i], _ = f.associate(z[i], R[i])
                if j[i] >= 0:
                    f.update(j[i], z[i], R[i])
                else:
                    f.add_line(z[i], R[i])
            outs.append((j, f.end_scan(len(z))[1]))
        self.x_t0 = None
        assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1]), s
        self.J.append(outs[0][0])

    def insert(self, lines, cov):
        k = len(lines)
        L = self.f.insert_lines(lines, cov) - k          # first: nothing reads the state of `f` before the call
        pose = self.f.pose                                # the insertion leaves the pose as it was
        y, P, Lg = self.g.download_live()
        assert Lg == L
        ye, Pe = np_insert(y, P, lines, cov)
        self.g.upload(*layout(ye, Pe, self.g.n), L + k)
        self.x_t0 = pose
        a, b = self.f.download_live(), self.g.download_live()
        assert a[2] == b[2] == L + k
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])

    def same(self, what):
        a, b = self.f.download_live(), self.g.download_live()
        assert a[2] == b[2], what
        assert np.array_equal(a[0], b[0]), what
        assert np.array_equal(a[1], b[1]), (what, np.argwhere(a[1] != b[1])[:5])

    def close(self):
        self.f.close(); self.g.close()


def observed_lines(t, scans):
    """World lines of the landmarks the given scans observe (landmark j = world line j while nothing moved)."""
    ids = sorted(set(int(w) for s in scans for w in t.scn["idx"][s]))
    return t.scn["world"][ids], ids


def test_insert_equals_upload_default(libekf):
    """3 300 landmarks, grouped overlapped scans.  Insertions: inside an open sweep group (after five scans); right after
    a ten-scan ekf_scan_device burst with no sync; as remove -> insert -> observe_pose; before chunked scans of 40 lines;
    before step-wise scans; and before scans of unmatched lines whose appends trigger the map reset (on both at the
    same scan).  At least 100 scans follow the last insertion."""
    import torch
    from slam_ros_b200 import scenario as sc
    N, cap = 3300, 3600
    t = Twins(N, cap, seed=23)
    rng = np.random.default_rng(29)
    for s in range(5):
        t.scan(s)
    lines, _ = observed_lines(t, range(5, 25))       # duplicates of existing landmarks: gated, never the first fit
    t.insert(lines[:20], spd(20, rng))
    for s in range(5, 25):
        t.scan(s)
    dev = torch.device("cuda")
    scn = t.scn
    d_u = torch.tensor(scn["u"], device=dev); d_z = torch.tensor(scn["z"], device=dev); d_R = torch.tensor(scn["R"], device=dev)
    d_j = {id(f): torch.zeros((10, 8), dtype=torch.int32, device=dev) for f in (t.f, t.g)}
    for f in (t.f, t.g):
        for i, s in enumerate(range(25, 35)):
            f.scan_device(d_u[s].data_ptr(), 8, d_z[s].data_ptr(), d_R[s].data_ptr(), d_j[id(f)][i].data_ptr())
    t.insert(random_lines(10, rng), None)             # waits for the burst itself
    assert torch.equal(d_j[id(t.f)], d_j[id(t.g)])
    for s in range(35, 55):
        t.scan(s)
    # remove -> insert -> observe_pose: the landmarks the next scans observe come back at the end of the map with their
    # marginal covariance, and the next scans match them there
    y, P, L = t.f.download_live()
    ids = sorted(set(int(w) for s in range(55, 70) for w in scn["idx"][s]))
    si = np.array([3 + 2 * j + q for j in ids for q in (0, 1)])
    for f in (t.f, t.g):
        assert f.remove_lines(ids) == L - len(ids)
    t.insert(y[si].reshape(-1, 2), P[np.ix_(si, si)])
    zf, Rf = t.f.pose + np.array([2e-3, -1e-3, 1e-3]), np.diag([1e-4, 1e-4, 1e-5])
    for f in (t.f, t.g):
        f.observe_pose(zf, Rf)
    t.x_t0 = None
    t.same("after remove -> insert -> observe_pose")
    Lr = t.f.lines
    J = [t.scan(s) for s in range(55, 70)]
    hits = sum(int((j >= Lr - len(ids)).sum()) for j in J)
    assert hits >= 90, "only %d of the 120 lines matched the re-inserted landmarks" % hits
    t.insert(random_lines(12, rng), spd(12, rng))
    for s in range(70, 75):                           # chunked: 40 lines per scan
        ids40 = (7 * s + np.arange(40)) % N
        z = sc.observe(scn["world"][ids40], scn["poses"][s + 1]) + rng.standard_normal((40, 2)) * 1e-4
        z[:, 0] = sc.wrap_pi(z[:, 0])
        t.scan(s, z, sc.declared_R(40))
    t.insert(random_lines(6, rng), None)
    for s in range(75, 80):
        t.stepwise(s)
    for s in range(80, 95):
        t.scan(s)
    t.same("scan 94")
    L = t.f.lines
    k = cap - 10 - L - 12                             # two scans of eight unmatched lines pass cap - headroom
    t.insert(random_lines(k, rng), spd(k, rng, 1e-6))
    L_before = t.f.lines
    reset_at = None
    for s in range(95, 220):
        z = scn["z"][s].copy()
        if s < 99:
            z[:, 1] += 3.0 + 0.25 * (s - 95)          # unmatched: appended
        t.scan(s, z)
        if reset_at is None and t.f.lines < L_before:
            reset_at = s
        L_before = t.f.lines
    assert reset_at is not None and reset_at <= 97, reset_at
    t.same("end")
    t.close()


@pytest.mark.parametrize("max_batch", [1, 16])
def test_insert_equals_upload_max_batch(libekf, max_batch):
    """max_batch = 1 and 16 (one pending slot, and a flush inside every 8-line scan pair's pending list): insertion
    after three scans, then 100 scans; halfway a second insertion with a prior block."""
    rng = np.random.default_rng(31 + max_batch)
    t = Twins(3300, 3400, seed=37, max_batch=max_batch, S=110)
    for s in range(3):
        t.scan(s)
    lines, _ = observed_lines(t, range(3, 20))
    t.insert(lines[:16], None)
    for s in range(3, 103):
        t.scan(s)
        if s == 50:
            t.insert(random_lines(24, rng), spd(24, rng))
    t.same("end")
    t.close()


# ---- 3. surveyed landmarks stay fixed on every path -----------------------------------------------------------------
# path -> (environment, flags, entry, big map)
PATHS = {
    "stepwise": ({}, 0, "stepwise", False),
    "fused": ({}, 0, "scan", False),
    "line_loop1": ({"EKF_LINE_LOOP": "1"}, 0, "scan", False),
    "per_line": ({}, 4, "scan", False),
    "eager": ({}, 1, "scan", False),
    "overlap": ({}, 0, "scan", True),
    "no_overlap": ({}, 8, "scan", True),
    "chunked": ({}, 0, "chunked", True),
    "device": ({}, 0, "device", True),
    "device_small": ({}, 0, "device", False),
}


def surveyed_run(path):
    """Runs in a subprocess (environment knobs are read once per process).  Returns the list of failures."""
    from slam_ros_b200 import EkfFilter
    env, flags, entry, big = PATHS[path]
    L0, cap = (3000, 3060) if big else (12, 40)
    rng = np.random.default_rng(sum(map(ord, path)))
    y, P, world = hp.spread_state(L0, cap, 17, decades=(-4.0, -2.0))
    f = EkfFilter(capacity_lines=cap, reset_headroom=0, flags=flags)
    f.upload(y, P, L0)
    k = 4
    walls = random_lines(k, rng, r=(9.5, 12.0))
    assert f.insert_lines(walls, None) == L0 + k
    wall_y = f.download_y()[3 + 2 * L0:]
    allw = np.concatenate([world, walls])
    ins = list(range(L0, L0 + k))
    pose = tuple(y[:3])
    fails = []
    m_old = 36 if entry == "chunked" else 4
    n_scans = 12

    def check(what, j):
        yy = f.download_y()
        nl = yy.size
        if not np.array_equal(yy[3 + 2 * L0:3 + 2 * (L0 + k)], wall_y):
            fails.append("%s: the surveyed landmarks' y changed" % what)
        B = f.download_block(3 + 2 * L0, 0, 2 * k, nl)
        if (B != 0).any():
            fails.append("%s: %d nonzero entries in the surveyed rows of P (max %.3g)" % (what, int((B != 0).sum()), np.abs(B).max()))
        if j is not None and not np.array_equal(j[:k], ins):
            fails.append("%s: the surveyed walls matched %s" % (what, j[:k]))

    def lines(s):
        nonlocal pose
        pose = hp.predicted_pose(pose, U)
        ids = ins + [int(i) for i in rng.choice(L0, m_old, replace=False)]
        return hp.lines_for(allw, pose, ids, rng, n_unmatched=1 if s % 3 == 0 else 0)

    for s in range(n_scans):
        z, R = lines(s)
        if entry == "stepwise":
            f.predict(np.array(U))
            j = np.full(len(z), -1, np.int32)
            for i in range(len(z)):
                j[i], _ = f.associate(z[i], R[i])
                if j[i] >= 0:
                    f.update(j[i], z[i], R[i])
                else:
                    f.add_line(z[i], R[i])
            f.end_scan(len(z))
        elif entry == "device":
            import torch
            du, dz, dR = (torch.tensor(np.ascontiguousarray(a), device="cuda") for a in (np.array(U), z, R))
            dj = torch.full((len(z),), -7, dtype=torch.int32, device="cuda")
            f.scan_device(du.data_ptr(), len(z), dz.data_ptr(), dR.data_ptr(), dj.data_ptr())
            f.sync()
            j = dj.cpu().numpy()
        else:
            j = f.scan(np.array(U), z, R)[1]
        check("%s scan %d" % (path, s), j)
    if big:                                          # scans in a row with no read in between: sweep groups stay open
        for s in range(n_scans, n_scans + 8):
            z, R = lines(s)
            j = f.scan(np.array(U), z, R)[1]
            if not np.array_equal(j[:k], ins):
                fails.append("%s scan %d: the surveyed walls matched %s" % (path, s, j[:k]))
        check("%s after 8 unread scans" % path, None)
    if big and 3 + 2 * f.lines < OVERLAP_MIN_N:
        fails.append("%s: the map fell below the overlapped path's size" % path)
    f.close()
    return fails


def _spawn(call, env_extra):
    code = "import sys; sys.path[:0] = [%r, %r]\nimport test_gpu_insert_lines as t\nr = %s\nprint('FAILS', repr(r))\n" % (
        ROOT, TESTS, call)
    env = dict(os.environ)
    for k in ("EKF_LINE_LOOP", "EKF_LIB", "EKF_CHUNK", "EKF_CHUNK_ABOVE", "EKF_SWEEP_GROUP"):
        env.pop(k, None)
    env.update(env_extra)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=1200, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("FAILS ")][-1]
    return eval(line[6:])


@pytest.mark.parametrize("path", list(PATHS))
def test_surveyed_landmarks_stay_fixed(libekf, path):
    fails = _spawn("t.surveyed_run(%r)" % path, PATHS[path][0])
    assert not fails, fails[:4]


# ---- 4. against the structured oracle --------------------------------------------------------------------------------
def wall_lines(walls):
    """World (alfa, r) of wall segments (x0, y0, x1, y1): x cos(alfa) + y sin(alfa) = r, r >= 0, alfa in (-pi, pi];
    segments on one line give one landmark."""
    out = []
    for x0, y0, x1, y1 in walls:
        dx, dy = x1 - x0, y1 - y0
        nx, ny = -dy / math.hypot(dx, dy), dx / math.hypot(dx, dy)
        r = nx * x0 + ny * y0
        if r < 0:
            nx, ny, r = -nx, -ny, -r
        a = math.atan2(ny, nx)
        if not any(abs(a - b) < 1e-9 and abs(r - q) < 1e-9 for b, q in out):
            out.append((a, r))
    return np.array(out)


def oracle_insert(o, lines, cov):
    y = np.ctypeslib.as_array(o._lib.ekfo_y_ptr(o._h), shape=(o.n,))
    P = o.P_view()
    L = o.lines
    nl0, k = 3 + 2 * L, len(lines)
    nl = nl0 + 2 * k
    y[nl0:nl] = np.asarray(lines, np.float64).ravel()
    P[nl0:nl, :nl] = 0.0
    P[:nl, nl0:nl] = 0.0
    if cov is not None:
        P[nl0:nl, nl0:nl] = cov
    o._lib.ekfo_set_lines(o._h, C.c_int(L + k))


def oracle_remove(o, removed):
    """Removal on the oracle in numpy, as tests/test_gpu_remove_lines.py does it."""
    L = o.lines
    gone = set(int(j) for j in removed)
    keep = np.array([0, 1, 2] + [3 + 2 * j + t for j in range(L) if j not in gone for t in (0, 1)])
    nl, nl_old = keep.size, 3 + 2 * L
    y = np.ctypeslib.as_array(o._lib.ekfo_y_ptr(o._h), shape=(o.n,))
    P = o.P_view()
    ynew, Pnew = y[keep].copy(), P[np.ix_(keep, keep)].copy()
    y[:nl] = ynew; y[nl:nl_old] = 0.0
    P[:nl, :nl] = Pnew; P[nl:nl_old, :nl_old] = 0.0; P[:nl_old, nl:nl_old] = 0.0
    o._lib.ekfo_set_lines(o._h, C.c_int(L - len(removed)))


def _close(f, o, what):
    y, P, L = f.download_live()
    yo, Po = o.live()
    assert L == o.lines, what
    assert np.abs(y - yo).max() <= 1e-9 * max(np.abs(yo).max(), 1e-300), what
    assert np.abs(P - Po).max() <= 1e-9 * np.abs(Po).max(), what


def test_floor_plan_against_oracle(libekf):
    """The room's walls inserted as a surveyed floor plan on a fresh filter, then 200 room scans: associations
    bit-exact, y and P within 1e-9 after every scan, hundreds of lines matched to the floor plan before the map reset
    drops it."""
    from oracle.oracle import StructuredOracle
    from slam_ros_b200 import EkfFilter, scenario as sc
    walls = wall_lines(sc.room_walls())
    assert 15 <= len(walls) <= 20
    cap, S = 200, 200
    scn = sc.room_scenario(steps=S)
    f = EkfFilter(capacity_lines=cap)
    o = StructuredOracle(cap, threads=0)
    assert f.insert_lines(walls) == len(walls)
    oracle_insert(o, walls, None)
    _close(f, o, "after the insertion")
    on_plan, reset_at = 0, None
    for s in range(S):
        c = int(scn["count"][s])
        z, R = scn["z"][s, :c], scn["R"][s, :c]
        L = o.lines
        J = f.scan(scn["u"][s], z, R)[1]
        st, Jo = o.scan(scn["u"][s], z, R)
        assert np.array_equal(J, Jo), s
        _close(f, o, "scan %d" % s)
        if reset_at is None and o.lines < L:
            reset_at = s
        if reset_at is None:
            on_plan += int(((J >= 0) & (J < len(walls))).sum())
    # lines fitted to a partition seen from its far side, or to part of a wall, are appended as SLAM landmarks; the map
    # reset then drops the floor plan with them
    assert on_plan >= 300 and reset_at is not None, (on_plan, reset_at)
    f.close(); o.close()


def test_prior_block_mid_run_against_oracle(libekf):
    """3 300 landmarks; after 11 scans (a sweep group open) the landmarks the next scans observe are removed and
    inserted again at the end of the map with their marginal covariance as the prior block; 60 scans follow."""
    from oracle.oracle import StructuredOracle
    from slam_ros_b200 import EkfFilter, scenario as sc
    N, cap, S = 3300, 3400, 71
    scn = sc.map_scenario(N, S, m=8, seed=43)
    f = EkfFilter(capacity_lines=cap)
    o = StructuredOracle(cap, threads=0)
    f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"]); o.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])

    def run(s):
        J = f.scan(scn["u"][s], scn["z"][s], scn["R"][s])[1]
        Jo = o.scan(scn["u"][s], scn["z"][s], scn["R"][s])[1]
        assert np.array_equal(J, Jo), s
        return J

    for s in range(11):
        run(s)
    ids = sorted(set(int(w) for s in range(11, 31) for w in scn["idx"][s]))
    y, P, L = f.download_live()
    si = np.array([3 + 2 * j + q for j in ids for q in (0, 1)])
    lines, cov = y[si].reshape(-1, 2), P[np.ix_(si, si)]
    cov = np.triu(cov) + np.triu(cov, 1).T
    assert f.remove_lines(ids) == L - len(ids)
    oracle_remove(o, ids)
    assert f.insert_lines(lines, cov) == L
    oracle_insert(o, lines, cov)
    _close(f, o, "after the insertion")
    matched = 0
    for s in range(11, S):
        J = run(s)
        matched += int((J >= L - len(ids)).sum())
        if s % 10 == 0 or s == S - 1:
            _close(f, o, "scan %d" % s)
    assert matched >= len(ids), matched
    f.close(); o.close()


# ---- 5. componentwise against the extended-precision reference --------------------------------------------------------
def _sym3(T):
    A = np.array(T[:, :3])
    return np.triu(A) + np.triu(A, 1).T


def test_insert_lines_componentwise_continuation(libekf):
    """A spread state of 3 000 landmarks, six warm-up scans that leave pending terms in both halves of the slot ring,
    then 68 landmarks with a prior block inserted to nl = 6 139, just below the tile edge at 6 144.  The state goes into
    hp.HPFilter; then five sweep groups of two scans that observe inserted landmarks too, each appending two ghosts
    (9 m beyond a landmark; the inserted ones lie beyond those) in its first scan and matching them in its second, so
    the appends land beyond the inserted block and cross the tile edge."""
    from slam_ros_b200 import EkfFilter
    L0, cap, k = 3000, 3100, 68
    rng = np.random.default_rng(47)
    y, P, world = hp.spread_state(L0, cap, 47)
    f = EkfFilter(capacity_lines=cap, reset_headroom=0)
    f.upload(y, P, L0)
    pose = tuple(y[:3])
    warm = 0
    for _ in range(6):
        pose = hp.predicted_pose(pose, U)
        z, R = hp.lines_for(world, pose, rng.choice(L0, 8, replace=False), rng)
        warm += int((f.scan(np.array(U), z, R)[1] >= 0).sum())
    assert warm >= 32, warm
    ins = random_lines(k, rng, r=(20.0, 24.0))            # beyond every landmark and every ghost
    assert f.insert_lines(ins, spd(k, rng, 1e-4)) == L0 + k
    y1, P1, L1 = f.download_live()
    assert 3 + 2 * L1 == 6139
    wc = [tuple(w) for w in world] + [tuple(w) for w in ins]
    ref = hp.HPFilter(cap, reset_headroom=0)
    ref.upload(y1, P1, L1)
    pose = tuple(y1[:3])
    placed, fails = [], []
    for g in range(5):
        for first in (True, False):
            pose = hp.predicted_pose(pose, U)
            true_ids = [int(i) for i in rng.choice(L0, 4, replace=False)] + [L0 + int(i) for i in rng.choice(k, 2, replace=False)]
            if first:
                src = [int(i) for i in rng.integers(0, L0, 2)]
                wl = [wc[i] for i in true_ids] + [(wc[i][0], wc[i][1] + 9.0) for i in src]
            else:
                wl = placed + [wc[i] for i in true_ids]
            z, R = hp.lines_for(np.array(wl), pose, range(len(wl)), rng)
            if first:
                placed = [(float(np.mod(z[q, 0] + pose[2] + np.pi, 2 * np.pi) - np.pi),
                           z[q, 1] + pose[0] * np.cos(z[q, 0]) + pose[1] * np.sin(z[q, 0])) for q in (6, 7)]
            rc, J, xp = f.scan(np.array(U), z, R)
            st, Jr = ref.scan(np.array(U), z, R)
            if not np.array_equal(J, Jr):
                fails.append("group %d: associations %s vs %s" % (g, J, Jr))
            if first and not (J[4:6] >= L0).all():
                fails.append("group %d: the inserted landmarks were not matched: %s" % (g, J))
            if not first and not (J[:2] >= L1).all():
                fails.append("group %d: the ghosts of its first scan were not matched" % g)
            for what, x, v, m_ in (("pose", xp, ref.pose, ref.mpose), ("rcov", f.robot_cov(), _sym3(ref.T), _sym3(ref.mT))):
                w = hp.worst_ratio(np.asarray(x, np.float64), v, m_) / ref.C
                if w > 1.0:
                    fails.append("group %d %s: worst |x - ref| / (C u mag) = %.3g" % (g, what, w))
            if f.lines != ref.L:
                fails.append("group %d: %d lines vs %d" % (g, f.lines, ref.L))
    assert not fails, fails[:5]
    assert ref.min_margin >= 1e-6, ref.min_margin
    f.sync()
    nl = ref.nl
    assert nl > 6144 and nl == 3 + 2 * f.lines
    t = 64 * ((nl - 1) // 64)
    blocks = [(0, 0, 3, nl), (t, 0, nl - t, nl), (0, t, nl, nl - t), (6080, 6080, nl - 6080, nl - 6080)]
    blocks += [(d, d, min(64, nl - d), min(64, nl - d)) for d in range(0, nl, 64)]
    blocks += [(3 + 2 * j, 0, 2, nl) for j in range(L0, ref.L)]
    for _ in range(32):
        r0, c0 = (int(v) * 64 for v in rng.integers(0, (nl - 1) // 64 + 1, 2))
        blocks.append((r0, c0, min(64, nl - r0), min(64, nl - c0)))
    w = hp.worst_ratio(f.download_y(), ref.y[:nl], ref.my[:nl]) / ref.C
    assert w <= 1.0, "y: %.3g" % w
    for r0, c0, nr, nc in blocks:
        v, m_ = ref.block(np.arange(r0, r0 + nr), np.arange(c0, c0 + nc))
        w = hp.worst_ratio(f.download_block(r0, c0, nr, nc), v, m_) / ref.C
        assert w <= 1.0, "P block (%d, %d, %d, %d): %.3g" % (r0, c0, nr, nc, w)
    f.close()


# ---- 6. errors ---------------------------------------------------------------------------------------------------------
def test_insert_lines_errors_leave_state_unchanged(libekf):
    from slam_ros_b200 import scenario as sc
    from slam_ros_b200.ekf import EKF_EINVAL, EKF_ECAPACITY, EKF_ESTATE, EKF_OK
    cap = 3326
    f = seeded_map(3300, cap, 3)                        # three scans: a sweep group is open
    lib = f._lib
    L = f.lines
    rng = np.random.default_rng(53)
    dp = C.POINTER(C.c_double)

    def call(lines, cov=None, k=None):
        la = None if lines is None else np.ascontiguousarray(lines, dtype=np.float64)
        ca = None if cov is None else np.ascontiguousarray(cov, dtype=np.float64)
        n = C.c_int(-5)
        kk = (0 if la is None else la.size // 2) if k is None else k
        rc = lib.ekf_insert_lines(f.handle, kk, None if la is None else la.ctypes.data_as(dp),
                                  None if ca is None else ca.ctypes.data_as(dp), C.byref(n))
        return rc, n.value

    good = random_lines(3, rng)
    cov = spd(3, rng)
    before = f.download_live() + (f.pose, f.robot_cov())
    assert call(good, k=-1)[0] == EKF_EINVAL
    assert call(None, k=2)[0] == EKF_EINVAL
    for bad in (np.nan, np.inf, -np.inf):
        for pos in ((0, 0), (2, 1)):
            ln = good.copy(); ln[pos] = bad
            assert call(ln)[0] == EKF_EINVAL, (bad, pos)
    c = cov.copy(); c[1, 4] = np.nextafter(c[1, 4], 1.0)
    assert call(good, c)[0] == EKF_EINVAL                       # one ulp from symmetric
    for bad in (np.nan, np.inf):
        c = cov.copy(); c[0, 5] = c[5, 0] = bad
        assert call(good, c)[0] == EKF_EINVAL, bad
        c = cov.copy(); c[3, 3] = bad
        assert call(good, c)[0] == EKF_EINVAL, bad
    c = cov.copy(); c[4, 4] = -1e-30
    assert call(good, c)[0] == EKF_EINVAL
    big = random_lines(cap - L + 1, rng)
    assert call(big)[0] == EKF_ECAPACITY
    assert call(big, spd(cap - L + 1, rng))[0] == EKF_ECAPACITY
    assert call(np.zeros((0, 2))) == (EKF_OK, L)
    after = f.download_live() + (f.pose, f.robot_cov())
    assert after[2] == before[2] == L
    assert all(np.array_equal(a, b) for i, (a, b) in enumerate(zip(before, after)) if i != 2)
    scn = sc.map_scenario(3300, 1, m=8, seed=11)
    f.predict(scn["u"][0])
    assert call(good)[0] == EKF_ESTATE
    f.end_scan(0)
    assert f.lines == L
    # a zero diagonal (surveyed entries inside a prior block) is accepted
    c = cov.copy(); c[2, :] = 0.0; c[:, 2] = 0.0
    assert call(good, c) == (EKF_OK, L + 3)
    assert call(random_lines(cap - L - 3, rng)) == (EKF_OK, cap)
    f.close()


def test_insert_lines_row_sharded_is_refused(libekf):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29533",
           os.path.join(ROOT, "tests", "multi_gpu", "insert_sharded_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert out.stdout.count("insert_lines refused") == 2


# ---- 7. the mirrors ----------------------------------------------------------------------------------------------------
def test_python_robot_insert_lines(libekf):
    from slam_ros_b200 import scenario as sc
    from slam_ros_b200.robot import Robot
    rob = Robot(0.0, 0.0, 0.0, linesize=50)
    walls = wall_lines(sc.room_walls())
    assert rob.insert_lines(walls) == rob.savedLineCount == len(walls)
    assert rob.insert_lines(walls[:2], np.eye(4) * 1e-4) == len(walls) + 2
    rob.filter.close()


def test_cpp_robot_insert_lines(libekf):
    """tests/cpp/insert_main.cpp: ekfcuda::Robot inserts ten surveyed walls before its first localize; every line then
    matches them and savedLineCount stays; errors throw and leave it; a reset drops the walls and they go back in."""
    from slam_ros_b200 import library_path
    with tempfile.TemporaryDirectory() as d:
        exe = os.path.join(d, "insert")
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([cxx, "-std=c++11", "-O2", "-I", os.path.join(ROOT, "include"),
                               os.path.join(ROOT, "tests", "cpp", "insert_main.cpp"), library_path(),
                               "-Wl,-rpath," + os.path.dirname(library_path()), "-o", exe])
        out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "insert_main OK" in out.stdout, out.stdout
