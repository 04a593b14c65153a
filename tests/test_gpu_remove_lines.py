"""ekf_remove_lines: landmarks removed from a resident map (exact marginalisation: their entries of y and their rows and
columns of P are deleted, the later landmarks move down in order).

1. Bitwise against numpy deletion on the downloaded state, on the out-of-place path (second covariance buffer) and the
   in-place path (EKF_FLAG_NO_OVERLAP), which must also agree with each other bit for bit.
2. Continuation against the structured CPU oracle, which removes the same landmarks in numpy: associations bit-exact for
   every line over more than 100 scans, y and P within 1e-9, with the removal inside an open sweep group, after a
   device-resident burst and before the appends that trigger the map reset.
3. Componentwise against the extended-precision reference after a removal, on grouped overlapped scans that append into
   the vacated rows across a tile boundary (stale pending-slot rows would show there).
4. The same removal-and-continue sequence with one sweep per scan (EKF_SWEEP_GROUP=0) and grouped: identical bits.
5. Errors leave the state bitwise unchanged.
6. The C++ mirror (include/ekf_robot.hpp): Robot::removeLines.
"""
import ctypes as C
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


def keep_index(L, removed):
    """Old state index of every kept state entry, in the new order."""
    gone = set(int(j) for j in removed)
    kept = [j for j in range(L) if j not in gone]
    return np.array([0, 1, 2] + [3 + 2 * j + t for j in kept for t in (0, 1)], dtype=np.int64)


def state_index(removed):
    return np.array([3 + 2 * int(j) + t for j in removed for t in (0, 1)], dtype=np.int64)


def seeded_map(N, cap, steps, flags=0, seed=11):
    from slam_ros_b200 import EkfFilter, scenario as sc
    scn = sc.map_scenario(N, steps, m=8, seed=seed)
    f = EkfFilter(capacity_lines=cap, flags=flags)
    f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    for s in range(steps):
        f.scan(scn["u"][s], scn["z"][s], scn["R"][s])
    return f


def removal_sets(L, rng):
    """name -> strictly increasing landmark indices, for a map of L landmarks."""
    j64 = (64 * 3 - 3) // 2 - 3            # rows 3 + 2 j of these six landmarks straddle row 192 (a 64-row tile edge)
    sets = {
        "first": [0], "last": [L - 1], "none": [], "every_other": list(range(0, L, 2)),
        "tile_block": list(range(j64, j64 + 6)),
        "random10": sorted(rng.choice(L, L // 10, replace=False).tolist()),
    }
    for res in (1, 63):                     # nl' = 3 + 2 (L - k) = res (mod 64)
        k = (L - (res - 3) % 64 // 2) % 32 + 32
        sets["nl%d" % res] = sorted(rng.choice(L, k, replace=False).tolist())
    sets["all"] = list(range(L))
    return sets


# ---- 1. bitwise against numpy ---------------------------------------------------------------------------------------
def test_remove_lines_bitwise_against_numpy_3300(libekf):
    """3 300 landmarks (overlapped path, n >= 6000), capacity 3 326 (n = 6 655 = 255 mod 256): every removal set on a
    fresh copy of the same state, on both paths."""
    from slam_ros_b200.ekf import EKF_FLAG_NO_OVERLAP
    N, cap = 3300, 3326
    fs = {"oop": seeded_map(N, cap, 5), "inplace": seeded_map(N, cap, 5, flags=EKF_FLAG_NO_OVERLAP)}
    y0, P0, L0 = fs["oop"].download_live()
    assert L0 == fs["inplace"].lines == N and 3 + 2 * L0 >= OVERLAP_MIN_N
    Y, P = np.zeros(cap * 2 + 3), np.zeros((cap * 2 + 3, cap * 2 + 3))
    Y[:y0.size] = y0; P[:y0.size, :y0.size] = P0
    sets = removal_sets(L0, np.random.default_rng(3))
    for name, idx in sets.items():
        si = state_index(idx)
        ye = np.delete(y0, si); Pe = np.delete(np.delete(P0, si, 0), si, 1)
        if name in ("nl1", "nl63"):
            assert ye.size % 64 == int(name[2:])
        got = {}
        for path, f in fs.items():
            f.upload(Y, P, L0)
            pose0, rcov0 = f.pose, f.robot_cov()
            Ln = f.remove_lines(idx)
            y, Pn, L = f.download_live()
            assert Ln == L == L0 - len(idx), (name, path)
            assert np.array_equal(y, ye), (name, path)
            assert np.array_equal(Pn, Pe), (name, path, np.argwhere(Pn != Pe)[:5])
            assert np.array_equal(f.pose, pose0) and np.array_equal(f.robot_cov(), rcov0), (name, path)
            got[path] = (y, Pn)
        assert all(np.array_equal(a, b) for a, b in zip(got["oop"], got["inplace"])), name
    for f in fs.values():
        f.close()


def test_remove_lines_bitwise_against_numpy_12000(libekf):
    """12 000 landmarks, capacity 12 030 (n = 24 063 = 255 mod 256): the in-place path takes many stage batches.  The
    removals are applied one after the other on the same map; each is checked on y, the robot rows and a set of
    64 x 64 blocks against the same blocks gathered from the state before it."""
    from slam_ros_b200.ekf import EKF_FLAG_NO_OVERLAP
    N, cap = 12000, 12030
    fs = {"oop": seeded_map(N, cap, 3), "inplace": seeded_map(N, cap, 3, flags=EKF_FLAG_NO_OVERLAP)}
    rng = np.random.default_rng(5)
    L = N
    order = ["first", "none", "tile_block", "random10", "nl1", "last", "nl63", "every_other", "all"]
    for name in order:
        idx = removal_sets(L, rng)[name]
        keep = keep_index(L, idx)
        nl = keep.size
        edges = sorted({0, max(nl - 64, 0), 128, 192 - 32} | {int(v) * 64 for v in rng.integers(0, max(nl // 64, 1), 12)})
        spots = [(r, c) for r in edges for c in edges if r <= c and r < nl and c < nl]
        got = {}
        for path, f in fs.items():
            y_old = f.download_y()
            top_old = f.download_block(0, 0, 3, y_old.size)
            pose0, rcov0 = f.pose, f.robot_cov()
            exp_blocks = []
            for r0, c0 in spots:
                nr, nc = min(64, nl - r0), min(64, nl - c0)
                rr, cc = keep[r0:r0 + nr], keep[c0:c0 + nc]
                B = f.download_block(int(rr[0]), int(cc[0]), int(rr[-1] - rr[0] + 1), int(cc[-1] - cc[0] + 1))
                exp_blocks.append(B[np.ix_(rr - rr[0], cc - cc[0])])
            Ln = f.remove_lines(idx)
            assert Ln == f.lines == L - len(idx), (name, path)
            y = f.download_y()
            assert np.array_equal(y, y_old[keep]), (name, path)
            top = f.download_block(0, 0, 3, nl)
            assert np.array_equal(top, top_old[:, keep]), (name, path)
            blocks = [f.download_block(r0, c0, min(64, nl - r0), min(64, nl - c0)) for r0, c0 in spots]
            for (r0, c0), B, E in zip(spots, blocks, exp_blocks):
                assert np.array_equal(B, E), (name, path, r0, c0)
            assert np.array_equal(f.pose, pose0) and np.array_equal(f.robot_cov(), rcov0), (name, path)
            got[path] = [y, top] + blocks
        assert all(np.array_equal(a, b) for a, b in zip(got["oop"], got["inplace"])), name
        L -= len(idx)
    assert L == 0
    for f in fs.values():
        f.close()


# ---- 2. continuation against the structured oracle ------------------------------------------------------------------
def oracle_remove(o, removed):
    """The same removal on the CPU oracle, in numpy through its y and P views; the vacated tail is zeroed as the
    oracle's map reset leaves it."""
    L = o.lines
    keep = keep_index(L, removed)
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


def test_remove_lines_continuation_against_oracle(libekf):
    """3 300 landmarks, m = 8, 160 scans after the first removal.  Removal 1 after 5 scans (a sweep group is open);
    removal 2 right after a 10-scan ekf_scan_device burst, with no sync in between; removal 3 followed by scans of
    unmatched lines whose appends trigger the map reset, which must happen at the same scan on both sides.  Removals 1
    and 2 include the landmarks the following scans observe, so those world lines are re-observed and re-appended."""
    import torch
    from oracle.oracle import StructuredOracle
    from slam_ros_b200 import EkfFilter, scenario as sc
    N, cap, S = 3300, 3600, 165                    # the reset fires once L > 3 590: only the ghost scans get there
    scn = sc.map_scenario(N, S, m=8, seed=23)
    z = scn["z"].copy()
    ghost = set()                                  # scans 95 .. the reset: every line 3 m (+ 0.25 m per scan) out
    f = EkfFilter(capacity_lines=cap)
    o = StructuredOracle(cap, threads=0)
    f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"]); o.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    rng = np.random.default_rng(29)
    world_of = list(range(N))                      # world line of every landmark of the map (-1: a ghost)
    resets = []

    def oracle_scan(s):
        L_before = o.lines
        st, jo = o.scan(scn["u"][s], z[s], scn["R"][s])
        world_of.extend(-1 if s in ghost else int(scn["idx"][s][i]) for i in range(8) if jo[i] < 0)
        if o.lines < L_before:
            resets.append(s)
            world_of[:] = []
        assert len(world_of) == o.lines
        return jo

    def run(s):
        if s >= 95 and not resets:
            ghost.add(s)
            z[s, :, 1] = scn["z"][s, :, 1] + 3.0 + 0.25 * (s - 95)
        J = f.scan(scn["u"][s], z[s], scn["R"][s])[1]
        assert np.array_equal(J, oracle_scan(s)), s
        assert f.lines == o.lines, s

    def pick(next_scans, extra):
        seen = set(int(w) for s in next_scans for w in scn["idx"][s])
        idx = set(j for j, w in enumerate(world_of) if w in seen)
        return sorted(idx | set(rng.choice(len(world_of), extra, replace=False).tolist()))

    def remove_both(idx):
        L = f.lines
        assert f.remove_lines(idx) == L - len(idx)
        oracle_remove(o, idx)
        gone = set(idx)
        world_of[:] = [w for j, w in enumerate(world_of) if j not in gone]
        assert f.lines == o.lines == len(world_of)
        _close(f, o, "after a removal")

    for s in range(5):                             # odd: the third sweep group is open at the removal
        run(s)
    idx1 = pick(range(5, 25), 100)
    remove_both(idx1)
    assert 3 + 2 * f.lines >= OVERLAP_MIN_N, f.lines
    for s in range(5, 45):
        run(s)
    _close(f, o, "scan 44")
    dev = torch.device("cuda")
    d_u = torch.tensor(scn["u"], device=dev); d_z = torch.tensor(z, device=dev); d_R = torch.tensor(scn["R"], device=dev)
    d_j = torch.zeros((10, 8), dtype=torch.int32, device=dev)
    for t, s in enumerate(range(45, 55)):
        f.scan_device(d_u[s].data_ptr(), 8, d_z[s].data_ptr(), d_R[s].data_ptr(), d_j[t].data_ptr())
    Jo = [oracle_scan(s) for s in range(45, 55)]   # the oracle runs the burst while the GPU still may
    idx2 = pick(range(55, 70), 40)
    L = len(world_of)
    assert f.remove_lines(idx2) == L - len(idx2)   # waits for the burst itself
    assert np.array_equal(d_j.cpu().numpy(), np.stack(Jo))
    oracle_remove(o, idx2)
    gone = set(idx2)
    world_of[:] = [w for j, w in enumerate(world_of) if j not in gone]
    _close(f, o, "after the burst's removal")
    for s in range(55, 95):
        run(s)
    _close(f, o, "scan 94")
    assert not resets
    remove_both(pick(range(95, 100), 16))
    for s in range(95, S):
        run(s)
    _close(f, o, "end")
    assert len(resets) == 1 and 95 < resets[0] < S - 5, resets
    assert len(idx1) > 100 and len(idx2) > 40
    f.close(); o.close()


# ---- 3. componentwise against the extended-precision reference --------------------------------------------------------
def _sym3(T):
    A = np.array(T[:, :3])
    return np.triu(A) + np.triu(A, 1).T


def test_remove_lines_componentwise_continuation(libekf):
    """A spread state of 3 100 landmarks (P over 8 decades), six warm-up scans that leave pending terms in both halves of
    the slot ring at every row, then 32 landmarks removed (landmark 0 among them: everything moves) to nl = 6 139, just
    below the tile edge at 6 144.  The compacted state goes into hp.HPFilter; then five sweep groups of two scans, each
    appending two ghosts in its first scan and matching them in its second, so appends reuse the vacated rows that still
    hold the warm-up's stale terms and cross the tile edge.  Between scans only hot storage is read."""
    from slam_ros_b200 import EkfFilter
    L0, cap, U = 3100, 3198, (0.02, 0.0, 0.01)
    rng = np.random.default_rng(31)
    y, P, world = hp.spread_state(L0, cap, 31)
    f = EkfFilter(capacity_lines=cap, reset_headroom=0)
    f.upload(y, P, L0)
    pose = tuple(y[:3])
    warm = 0
    for _ in range(6):
        pose = hp.predicted_pose(pose, U)
        z, R = hp.lines_for(world, pose, rng.choice(L0, 8, replace=False), rng)
        warm += int((f.scan(np.array(U), z, R)[1] >= 0).sum())
    assert warm >= 32, warm
    removed = [0] + sorted((1 + rng.choice(L0 - 1, 31, replace=False)).tolist())
    assert f.remove_lines(removed) == L0 - 32
    y1, P1, L1 = f.download_live()
    assert 3 + 2 * L1 == 6139
    kept = [j for j in range(L0) if j not in set(removed)]
    wc = [tuple(world[j]) for j in kept]
    ref = hp.HPFilter(cap, reset_headroom=0)
    ref.upload(y1, P1, L1)
    pose = tuple(y1[:3])
    placed, fails = [], []
    for g in range(5):
        for first in (True, False):
            pose = hp.predicted_pose(pose, U)
            true_ids = [int(i) for i in rng.choice(L1, 6, replace=False)]
            if first:
                src = [int(i) for i in rng.integers(0, L1, 2)]
                wl = [wc[i] for i in true_ids] + [(wc[i][0], wc[i][1] + 3.0) for i in src]
            else:
                wl = placed + [wc[i] for i in true_ids]
            z, R = hp.lines_for(np.array(wl), pose, range(len(wl)), rng)
            if first:
                placed = [(float(np.mod(z[k, 0] + pose[2] + np.pi, 2 * np.pi) - np.pi),
                           z[k, 1] + pose[0] * np.cos(z[k, 0]) + pose[1] * np.sin(z[k, 0])) for k in (6, 7)]
            rc, J, xp = f.scan(np.array(U), z, R)
            st, Jr = ref.scan(np.array(U), z, R)
            if not np.array_equal(J, Jr):
                fails.append("group %d: associations %s vs %s" % (g, J, Jr))
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
    blocks += [(3 + 2 * j, 0, 2, nl) for j in range(L1, ref.L)]
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


# ---- 4. sweep groups: one sweep per scan and grouped give the same bits --------------------------------------------
CHILD = r'''
import sys, numpy as np, torch
sys.path.insert(0, ROOT)
from slam_ros_b200 import EkfFilter, scenario as sc
N, cap, S = 3300, 3326, 40
scn = sc.map_scenario(N, S, m=8, seed=37)
f = EkfFilter(capacity_lines=cap)
f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
rng = np.random.default_rng(41)
J, X, L = [], [], []
def scan(s):
    rc, j, pose = f.scan(scn["u"][s], scn["z"][s], scn["R"][s]); J.append(j); X.append(pose); L.append(f.lines)
for s in range(5):
    scan(s)
seen = sorted(set(int(w) for s in range(5, 15) for w in scn["idx"][s]))          # landmark j = world line j so far
L.append(f.remove_lines(sorted(set(seen) | set(rng.choice(N, 50, replace=False).tolist()))))
for s in range(5, 20):
    scan(s)
dev = torch.device("cuda")
d_u = torch.tensor(scn["u"], device=dev); d_z = torch.tensor(scn["z"], device=dev); d_R = torch.tensor(scn["R"], device=dev)
d_j = torch.zeros((7, 8), dtype=torch.int32, device=dev)
for t, s in enumerate(range(20, 27)):
    f.scan_device(d_u[s].data_ptr(), 8, d_z[s].data_ptr(), d_R[s].data_ptr(), d_j[t].data_ptr())
L.append(f.remove_lines(sorted(rng.choice(f.lines, 40, replace=False).tolist())))
J.extend(d_j.cpu().numpy())
for s in range(27, S):
    scan(s)
f.sync()
y = f.download_y()
n = len(y)
spots = [(0, 0), (3, 3), (5, 900), (n - 64, n - 64), (0, n - 64), (n - 200, n - 64)]
np.savez(sys.argv[1], J=np.stack(J), X=np.stack(X), L=np.array(L), y=y, S=np.array(f.cov_stats()),
         B=np.stack([f.download_block(r0, c0, 64, 64) for r0, c0 in spots]))
'''.replace("ROOT", repr(ROOT))


def _child(group, tmp_path):
    path = os.path.join(str(tmp_path), "remove_group_%s.npz" % (group or "default"))
    env = dict(os.environ)
    env.pop("EKF_SWEEP_GROUP", None)
    if group is not None:
        env["EKF_SWEEP_GROUP"] = group
    out = subprocess.run([sys.executable, "-c", CHILD, path], capture_output=True, text=True, timeout=1200, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    return dict(np.load(path))


def test_remove_lines_sweep_groups_identical_bits(libekf, tmp_path):
    ref = _child("0", tmp_path)
    grp = _child(None, tmp_path)
    for k in sorted(ref):
        assert np.array_equal(ref[k], grp[k]), k
    assert (ref["J"][5:15] < 0).sum() >= 20            # the removed landmarks' lines were appended again
    assert 3 + 2 * ref["L"].min() >= OVERLAP_MIN_N      # every scan stayed on the overlapped path


# ---- 5. errors ---------------------------------------------------------------------------------------------------------
def test_remove_lines_errors_leave_state_unchanged(libekf):
    from slam_ros_b200 import scenario as sc
    from slam_ros_b200.ekf import EKF_EINVAL, EKF_ESTATE, EKF_OK
    f = seeded_map(3300, 3326, 3)                       # three scans: a sweep group is open
    lib = f._lib
    L = f.lines

    def call(lst, k=None):
        a = np.ascontiguousarray(np.asarray(lst, dtype=np.int32))
        n = C.c_int(-5)
        return lib.ekf_remove_lines(f.handle, len(lst) if k is None else k,
                                    a.ctypes.data_as(C.POINTER(C.c_int)) if lst else None, C.byref(n)), n.value

    before = f.download_live()
    for bad in ([3, 2], [5, 5], [-1], [L], [0, L + 7], [1, 2, 2, 3]):
        assert call(bad)[0] == EKF_EINVAL, bad
    assert call([1], k=-1)[0] == EKF_EINVAL
    assert lib.ekf_remove_lines(f.handle, 2, None, None) == EKF_EINVAL
    assert call([]) == (EKF_OK, L)
    after = f.download_live()
    assert all(np.array_equal(a, b) for a, b in zip(before[:2], after[:2])) and before[2] == after[2]
    scn = sc.map_scenario(3300, 1, m=8, seed=11)
    f.predict(scn["u"][0])
    assert call([0])[0] == EKF_ESTATE
    f.end_scan(0)
    assert f.lines == L
    f.close()


def test_remove_lines_row_sharded_is_refused(libekf):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29531",
           os.path.join(ROOT, "tests", "multi_gpu", "remove_sharded_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert out.stdout.count("remove_lines refused") == 2


# ---- 6. the C++ mirror ---------------------------------------------------------------------------------------------------
def test_cpp_robot_remove_lines(libekf):
    """tests/cpp/remove_main.cpp: ekfcuda::Robot runs room scans, removes landmarks, checks savedLineCount and that the
    next localize still runs (and re-appends the removed walls)."""
    from slam_ros_b200 import library_path
    with tempfile.TemporaryDirectory() as d:
        exe = os.path.join(d, "remove")
        cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
        subprocess.check_call([cxx, "-std=c++11", "-O2", "-I", os.path.join(ROOT, "include"),
                               os.path.join(ROOT, "tests", "cpp", "remove_main.cpp"), library_path(),
                               "-Wl,-rpath," + os.path.dirname(library_path()), "-o", exe])
        out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "remove_main OK" in out.stdout, out.stdout
