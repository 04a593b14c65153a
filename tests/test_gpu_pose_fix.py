"""ekf_observe_pose: an absolute pose measurement (x, y, theta or any subset) fused into a resident map on the device.

1. One fix of every mask, componentwise against an extended-precision evaluation of the same update from the state
   downloaded just before it (hp_reference's magnitudes and acceptance rule, C = pose_fix_ref.DEPTH_POSE): on an empty
   map, at sizes that put nl = 1 and 63 (mod 64), on the overlapped path (3 300 landmarks, n >= 6 000) with a sweep group open,
   and at 10 000 landmarks through download_block (robot rows, diagonal blocks, seeded 32 x 32 blocks).
2. Lockstep with the structured CPU oracle over 210 scans with a fix every few scans (noisy true poses, every mask):
   associations bit-exact on every line, y and P within 1e-9.  Fixes happen with a sweep group open, right after a
   device-resident burst, just before the appends that trigger the map reset, and next to remove_lines.
3. The same sequence gives identical bits in the default configuration, EKF_SWEEP_GROUP=0, EKF_FLAG_NO_OVERLAP,
   EKF_FLAG_SWEEP_DIRECT, EKF_LINE_LOOP=1 and max_batch = 1 (one pending slot: two one-term sweeps).
4. Gate: d2 is reported, d2_max = d2 accepts and the next double below rejects; a rejected fix and a singular S leave
   y and P bitwise unchanged.
5. Every error case leaves the state bitwise unchanged.
6. The mirrors: Python Robot.observe_pose + localize against the oracle, and the C++ Robot::observePose.
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
import pose_fix_ref as pf

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LD = np.longdouble
OVERLAP_MIN_N = 6000        # kOverlapMinN (ekf_api.cu)


def fix_R(rng):
    A = rng.standard_normal((3, 3)) * np.array([0.02, 0.02, 0.01])[:, None]
    R = A @ A.T + np.diag([1e-4, 1e-4, 4e-5])
    return np.triu(R) + np.triu(R, 1).T


def noisy(pose, rng):
    return np.asarray(pose, np.float64) + rng.standard_normal(3) * np.array([0.01, 0.01, 0.005])


def seeded_map(N, cap, steps, seed=11, **kw):
    from slam_ros_b200 import EkfFilter, scenario as sc
    f = EkfFilter(capacity_lines=cap, **kw)
    if N == 0:
        return f, None
    scn = sc.map_scenario(N, max(steps, 1), m=8, seed=seed)
    f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    for s in range(steps):
        f.scan(scn["u"][s], scn["z"][s], scn["R"][s])
    return f, scn


# ---- 1. componentwise -------------------------------------------------------------------------------------------------
def expected_fix(top, y, mask, z, R):
    """The fix in longdouble from the robot rows `top` (3 x nl, symmetrised) and y of the state before it.  Returns
    (K, KS, mK, mKS, y', my', d2) with hp_reference's magnitudes (formed from absolute values, as in HPFilter._update)."""
    sel = [c for c in range(3) if mask & (1 << c)]
    d = len(sel)
    PH = top[sel].T.astype(LD)
    S = PH[sel] + R[np.ix_(sel, sel)].astype(LD)
    Si = np.linalg.inv(np.asarray(S, np.float64)).astype(LD)
    for _ in range(3):
        Si = Si + Si @ (np.eye(d, dtype=LD) - S @ Si)
    v = z[sel].astype(LD) - y[sel].astype(LD)
    mv = np.abs(z[sel]) + np.abs(y[sel])
    for i, c in enumerate(sel):
        if c == 2:
            v[i], wc = hp.normalize_radian(v[i]); mv[i] += float(wc)
    aS, aSi, aPH = hp._f(S), hp._f(Si), hp._f(PH)
    K = PH @ Si; mK = aPH @ aSi + aPH @ (aSi @ aS @ aSi)
    KS = K @ S; mKS = mK @ aS
    y1 = y.astype(LD) + K @ v
    my1 = np.abs(y) + mK @ hp._f(v) + hp._f(K) @ mv
    y1[2], wc = hp.normalize_radian(y1[2]); my1[2] += float(wc)
    return K, KS, mK, mKS, y1, my1, float(v @ Si @ v)


def spots_for(nl, rng, k=24):
    """(r0, c0, nr, nc): the robot rows, the first and last diagonal 32 x 32 blocks, and k seeded 32 x 32 blocks."""
    last = max(nl - 32, 0)
    out = [(0, 0, 3, nl), (0, 0, min(32, nl), min(32, nl)), (last, last, nl - last, nl - last)]
    for _ in range(k):
        r0, c0 = sorted(int(v) for v in rng.integers(0, max(nl - 32, 1), 2))
        d = int(rng.integers(0, max(nl - 32, 1)))
        out += [(r0, c0, min(32, nl - r0), min(32, nl - c0)), (d, d, min(32, nl - d), min(32, nl - d))]
    return out


def check_one_fix(f, mask, rng, what):
    nl = 3 + 2 * f.lines
    y0 = f.download_y()
    top = f.download_block(0, 0, 3, nl)
    spots = spots_for(nl, rng)
    before = [f.download_block(*s) for s in spots]
    z = noisy(y0[:3], rng)
    R = fix_R(rng)
    K, KS, mK, mKS, y1, my1, d2r = expected_fix(top, y0, mask, z, R)
    rc, acc, d2, pose = f.observe_pose(z, R, mask=mask)
    assert rc == 0 and acc, (what, mask)
    assert abs(d2 - d2r) <= 1e-9 * max(d2r, 1.0), (what, mask, d2, d2r)
    C_ = pf.DEPTH_POSE
    worst = hp.check(f.download_y(), y1, my1, C_, "%s mask %d: y" % (what, mask)) / C_
    assert np.array_equal(pose, f.pose)
    for (r0, c0, nr, nc), B0 in zip(spots, before):
        r, c = np.arange(r0, r0 + nr), np.arange(c0, c0 + nc)
        exp = B0.astype(LD) - KS[r] @ K[c].T
        mag = np.abs(B0) + mKS[r] @ mK[c].T
        worst = max(worst, hp.check(f.download_block(r0, c0, nr, nc), exp, mag, C_,
                                    "%s mask %d: P block (%d, %d)" % (what, mask, r0, c0)) / C_)
    return worst


@pytest.mark.parametrize("case", ["empty", "nl1", "nl63", "overlapped", "10k"])
def test_pose_fix_componentwise(libekf, case):
    N, cap, steps = {"empty": (0, 40, 0), "nl1": (95, 140, 3), "nl63": (94, 140, 3),
                     "overlapped": (3300, 3326, 3), "10k": (10000, 10030, 3)}[case]
    f, _ = seeded_map(N, cap, steps)
    nl = 3 + 2 * f.lines
    if case == "nl1":
        assert nl % 64 == 1
    if case == "nl63":
        assert nl % 64 == 63
    if case in ("overlapped", "10k"):
        assert nl >= OVERLAP_MIN_N
    rng = np.random.default_rng(len(case))
    if case == "empty":                      # P[2,2] = 0 on a fresh filter: theta needs its own R_thth > 0
        worst = 0.0
        for mask in range(1, 8):
            g, _ = seeded_map(0, 40, 0)
            worst = max(worst, check_one_fix(g, mask, rng, case))
            g.close()
    else:                                    # each fix is checked against the state downloaded just before it
        worst = max(check_one_fix(f, mask, rng, case) for mask in range(1, 8))
    assert worst <= 1.0
    f.close()


# ---- 2. lockstep with the oracle ----------------------------------------------------------------------------------------
def _close(f, o, what):
    y, P, L = f.download_live()
    yo, Po = o.live()
    assert L == o.lines, what
    assert np.abs(y - yo).max() <= 1e-9 * max(np.abs(yo).max(), 1e-300), what
    assert np.abs(P - Po).max() <= 1e-9 * np.abs(Po).max(), what


def oracle_remove(o, removed):
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


def test_pose_fix_lockstep_with_oracle(libekf):
    """3 300 landmarks, m = 8, 210 scans, a fix every 3 scans rotating through the masks (odd scan counts: a sweep group
    is open at the fix); a fix right after a 10-scan ekf_scan_device burst, a fix next to remove_lines, and a fix just
    before ghost lines start the appends that reset the map (at the same scan on both sides)."""
    import torch
    from oracle.oracle import StructuredOracle
    from slam_ros_b200 import EkfFilter, scenario as sc
    N, cap, S = 3300, 3600, 210
    scn = sc.map_scenario(N, S, m=8, seed=23)
    poses = sc.true_trajectory(scn["u"])
    z = scn["z"].copy()
    f = EkfFilter(capacity_lines=cap)
    o = StructuredOracle(cap, threads=0)
    f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"]); o.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    rng = np.random.default_rng(29)
    nfix, resets = [0], []

    def fix(s):
        mask = 1 + nfix[0] % 7
        nfix[0] += 1
        zf, R = noisy(poses[s + 1], rng), fix_R(rng)
        rc, acc, d2, pose = f.observe_pose(zf, R, mask=mask)
        st, d2o, _, _ = pf.oracle_observe_pose(o, zf, R, mask)
        assert rc == 0 and acc and st == 1, (s, mask)
        assert abs(d2 - d2o) <= 1e-9 * max(d2o, 1.0), (s, d2, d2o)
        assert np.abs(pose - o.pose).max() <= 1e-9, (s, pose, o.pose)

    def run(s):
        if s >= 150 and not resets:
            z[s, :, 1] = scn["z"][s, :, 1] + 3.0 + 0.25 * (s - 150)
        L0 = o.lines
        J = f.scan(scn["u"][s], z[s], scn["R"][s])[1]
        st, jo = o.scan(scn["u"][s], z[s], scn["R"][s])
        assert np.array_equal(J, jo), s
        assert f.lines == o.lines, s
        if o.lines < L0:
            resets.append(s)

    for s in range(45):
        run(s)
        if s % 3 == 2:
            fix(s)
    _close(f, o, "scan 44")
    dev = torch.device("cuda")
    d_u = torch.tensor(scn["u"], device=dev); d_z = torch.tensor(z, device=dev); d_R = torch.tensor(scn["R"], device=dev)
    d_j = torch.zeros((10, 8), dtype=torch.int32, device=dev)
    for t, s in enumerate(range(45, 55)):
        f.scan_device(d_u[s].data_ptr(), 8, d_z[s].data_ptr(), d_R[s].data_ptr(), d_j[t].data_ptr())
    Jo = [o.scan(scn["u"][s], z[s], scn["R"][s])[1] for s in range(45, 55)]
    fix(54)                                  # right after the burst, with no sync in between
    assert np.array_equal(d_j.cpu().numpy(), np.stack(Jo))
    _close(f, o, "after the burst's fix")
    for s in range(55, 100):
        run(s)
        if s % 3 == 0:
            fix(s)
    removed = sorted(rng.choice(f.lines, 30, replace=False).tolist())
    fix(99)                                  # a fix, a removal, a fix
    assert f.remove_lines(removed) == o.lines - 30
    oracle_remove(o, removed)
    fix(99)
    _close(f, o, "around remove_lines")
    for s in range(100, 150):
        run(s)
        if s % 3 == 1:
            fix(s)
    fix(149)                                 # just before the appends that reset the map
    for s in range(150, S):
        run(s)
        if s % 4 == 0:
            fix(s)
    _close(f, o, "end")
    assert len(resets) == 1 and 150 < resets[0] < S - 5, resets
    assert nfix[0] >= 60
    f.close(); o.close()


# ---- 3. identical bits across configurations ------------------------------------------------------------------------------
CHILD = r'''
import sys, numpy as np, torch
sys.path.insert(0, ROOT)
from slam_ros_b200 import EkfFilter, scenario as sc
flags, max_batch = int(sys.argv[2]), int(sys.argv[3])
N, cap, S = 3300, 3600, 30
scn = sc.map_scenario(N, S, m=8, seed=37)
poses = sc.true_trajectory(scn["u"])
f = EkfFilter(capacity_lines=cap, flags=flags, max_batch=max_batch)
f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
rng = np.random.default_rng(41)
J, X, D = [], [], []
def fix(s, mask):
    A = rng.standard_normal((3, 3)) * 0.02
    R = A @ A.T + np.eye(3) * 1e-4
    R = np.triu(R) + np.triu(R, 1).T
    rc, acc, d2, pose = f.observe_pose(poses[s + 1] + rng.standard_normal(3) * 0.01, R, mask=mask)
    D.append(d2); X.append(pose)
for s in range(S):
    rc, j, pose = f.scan(scn["u"][s], scn["z"][s], scn["R"][s]); J.append(j); X.append(pose)
    if s % 2 == 0:
        fix(s, 1 + (s // 2) % 7)
dev = torch.device("cuda")
d_u = torch.tensor(scn["u"], device=dev); d_z = torch.tensor(scn["z"], device=dev); d_R = torch.tensor(scn["R"], device=dev)
for s in range(S - 6, S):
    f.scan_device(d_u[s].data_ptr(), 8, d_z[s].data_ptr(), d_R[s].data_ptr())
fix(S - 1, 7)
f.sync()
y = f.download_y()
n = len(y)
spots = [(0, 0), (3, 3), (5, 900), (n - 64, n - 64), (0, n - 64), (n - 200, n - 64)]
np.savez(sys.argv[1], J=np.stack(J), X=np.stack(X), D=np.array(D), y=y, S=np.array(f.cov_stats()),
         B=np.stack([f.download_block(r0, c0, 64, 64) for r0, c0 in spots]))
'''.replace("ROOT", repr(ROOT))


def _child(tmp_path, name, flags=0, max_batch=64, env_extra=None):
    path = os.path.join(str(tmp_path), "pose_%s.npz" % name)
    env = dict(os.environ)
    for k in ("EKF_SWEEP_GROUP", "EKF_LINE_LOOP"):
        env.pop(k, None)
    env.update(env_extra or {})
    out = subprocess.run([sys.executable, "-c", CHILD, path, str(flags), str(max_batch)], capture_output=True, text=True,
                         timeout=1200, env=env)
    assert out.returncode == 0, name + "\n" + out.stdout[-3000:] + out.stderr[-3000:]
    return dict(np.load(path))


def test_pose_fix_identical_bits_across_configurations(libekf, tmp_path):
    from slam_ros_b200.ekf import EKF_FLAG_NO_OVERLAP, EKF_FLAG_SWEEP_DIRECT
    ref = _child(tmp_path, "default")
    others = {"group0": _child(tmp_path, "group0", env_extra={"EKF_SWEEP_GROUP": "0"}),
              "no_overlap": _child(tmp_path, "no_overlap", flags=EKF_FLAG_NO_OVERLAP),
              "direct": _child(tmp_path, "direct", flags=EKF_FLAG_SWEEP_DIRECT),
              "line_loop1": _child(tmp_path, "line_loop1", env_extra={"EKF_LINE_LOOP": "1"}),
              "max_batch1": _child(tmp_path, "max_batch1", max_batch=1)}
    for name, got in others.items():
        for k in sorted(ref):
            assert np.array_equal(ref[k], got[k]), (name, k)
    assert (ref["J"] >= 0).mean() > 0.9 and ref["y"].size >= OVERLAP_MIN_N


# ---- 4. gate and rejection -------------------------------------------------------------------------------------------------
def test_pose_fix_gate_and_rejection(libekf):
    from slam_ros_b200.ekf import EKF_ESINGULAR
    f, _ = seeded_map(200, 260, 4)
    y0, P0, L0 = f.download_live()
    Y = np.zeros(f.n); Y[:y0.size] = y0
    Pf = np.zeros((f.n, f.n)); Pf[:y0.size, :y0.size] = P0
    rng = np.random.default_rng(3)
    z, R = noisy(y0[:3], rng), fix_R(rng)
    rc, acc, d2, _ = f.observe_pose(z, R, mask=7, d2_max=0.0)
    assert rc == 0 and not acc and d2 > 0
    y1, P1, _ = f.download_live()
    assert np.array_equal(y0, y1) and np.array_equal(P0, P1)
    f.upload(Y, Pf, L0)
    rc, acc, d2b, _ = f.observe_pose(z, R, mask=7, d2_max=np.nextafter(d2, 0))
    assert rc == 0 and not acc and d2b == d2
    y1, P1, _ = f.download_live()
    assert np.array_equal(y0, y1) and np.array_equal(P0, P1)
    f.upload(Y, Pf, L0)
    rc, acc, d2c, _ = f.observe_pose(z, R, mask=7, d2_max=d2)
    assert rc == 0 and acc and d2c == d2
    assert not np.array_equal(P0, f.download_live()[1])
    g, _ = seeded_map(0, 20, 0)                       # theta alone on a fresh filter: P[2,2] = 0, R_thth = 0
    yg, Pg, _ = g.download_live()
    rc, acc, d2, pose = g.observe_pose([0.0, 0.0, 0.3], np.zeros(9), mask=4)
    assert rc == EKF_ESINGULAR and not acc
    y1, P1, _ = g.download_live()
    assert np.array_equal(yg, y1) and np.array_equal(Pg, P1) and np.array_equal(pose, np.zeros(3))
    f.close(); g.close()


# ---- 5. errors ----------------------------------------------------------------------------------------------------------
def test_pose_fix_errors_leave_state_unchanged(libekf):
    from slam_ros_b200 import scenario as sc
    from slam_ros_b200.ekf import EKF_EINVAL, EKF_ESTATE, EKF_OK
    f, _ = seeded_map(3300, 3326, 3)                  # three scans: a sweep group is open
    lib = f._lib
    dp = C.POINTER(C.c_double)

    def call(mask, z, R, d2max=math.inf):
        za = None if z is None else np.ascontiguousarray(z, np.float64)
        Ra = None if R is None else np.ascontiguousarray(R, np.float64)
        d2 = C.c_double(-1); acc = C.c_int(-1); pose = np.zeros(3)
        return lib.ekf_observe_pose(f.handle, mask, None if za is None else za.ctypes.data_as(dp),
                                    None if Ra is None else Ra.ctypes.data_as(dp), C.c_double(d2max), C.byref(d2),
                                    C.byref(acc), pose.ctypes.data_as(dp))

    before = f.download_live()
    z = np.array([0.0, 0.0, 0.0]); R = np.eye(3).reshape(-1) * 1e-3
    asym = R.copy(); asym[1] = 1e-5                   # R[0][1] != R[1][0]
    for bad in [(0, z, R), (8, z, R), (-1, z, R), (7, None, R), (7, z, None),
                (7, np.array([np.nan, 0, 0]), R), (4, np.array([0, 0, np.inf]), R),
                (3, z, np.where(np.arange(9) == 4, np.nan, R)), (7, z, asym), (3, z, asym), (7, z, R, math.nan)]:
        assert call(*bad) == EKF_EINVAL, bad
    after = f.download_live()
    assert all(np.array_equal(a, b) for a, b in zip(before[:2], after[:2])) and before[2] == after[2]
    # entries outside the selection are not read: a NaN there and an asymmetric unselected pair are accepted
    assert call(3, np.array([0.0, 0.0, np.nan]), np.where(np.arange(9) == 8, np.nan, R), -1.0) == EKF_OK
    assert call(4, z, asym, -1.0) == EKF_OK           # d2_max < 0: rejected, nothing changes
    after = f.download_live()
    assert all(np.array_equal(a, b) for a, b in zip(before[:2], after[:2]))
    scn = sc.map_scenario(3300, 1, m=8, seed=11)
    L = f.lines
    f.predict(scn["u"][0])
    assert call(7, z, R) == EKF_ESTATE
    f.end_scan(0)
    assert f.lines == L
    f.close()


# ---- 6. mirrors --------------------------------------------------------------------------------------------------------------
def test_python_robot_observe_pose_then_localize(libekf):
    """Robot.observe_pose moves xPos / yPos / thetaPos, so the next localize predicts from the corrected pose: the same
    as pose_fix_ref.oracle_observe_pose + ekfo_localize on the oracle (odometry from (corrected pose - encoder))."""
    from oracle.oracle import StructuredOracle
    from slam_ros_b200 import Robot, Line, scenario as sc
    N, S = 60, 20
    scn = sc.map_scenario(N, S, m=8, seed=3)
    poses = sc.true_trajectory(scn["u"])
    rob = Robot(0.0, 0.0, 0.0, linesize=120)
    o = StructuredOracle(120)
    rng = np.random.default_rng(9)

    def lines(zz, RR):
        return [Line(float(a), float(r), tuple(RR[i])) for i, (a, r) in enumerate(zz)]

    enc = np.zeros(3)
    rob.localize(lines(scn["seed_z"], scn["seed_R"]), encoder=enc)
    o.localize(scn["seed_z"], scn["seed_R"], enc)
    for s in range(S):
        enc = poses[s] - np.array([scn["u"][s][0] * math.cos(poses[s][2]), scn["u"][s][0] * math.sin(poses[s][2]),
                                   scn["u"][s][2]])
        rob.localize(lines(scn["z"][s], scn["R"][s]), encoder=enc)
        st, jo = o.localize(scn["z"][s], scn["R"][s], enc)
        assert np.array_equal(rob.last_matches, jo), s
        if s % 3 == 1:
            zf, R = noisy(poses[s + 1], rng), fix_R(rng)
            rc, acc, d2 = rob.observe_pose(zf, R, mask=1 + s % 7)
            st, d2o, _, _ = pf.oracle_observe_pose(o, zf, R, 1 + s % 7)
            assert rc == 0 and acc and st == 1
        assert np.abs(np.array([rob.xPos, rob.yPos, rob.thetaPos]) - o.pose).max() <= 1e-9, s
    y, P, L = rob.filter.download_live()
    yo, Po = o.live()
    assert L == o.lines and np.abs(y - yo).max() <= 1e-9 * np.abs(yo).max()
    assert np.abs(P - Po).max() <= 1e-9 * np.abs(Po).max()
    o.close()


def test_cpp_robot_observe_pose(libekf):
    from slam_ros_b200 import library_path
    with tempfile.TemporaryDirectory() as d:
        exe = os.path.join(d, "pose_fix")
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([cxx, "-std=c++11", "-O2", "-I", os.path.join(ROOT, "include"),
                               os.path.join(ROOT, "tests", "cpp", "pose_fix_main.cpp"), library_path(),
                               "-Wl,-rpath," + os.path.dirname(library_path()), "-o", exe])
        out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "pose_fix_main OK" in out.stdout, out.stdout
