"""The two exceptional branches of Robot::localize on every scan path, against the extended-precision reference.

* A singular innovation covariance S: the pair is no match, first fit continues with the next landmark, and the scan
  reports EKF_ESINGULAR (include/ekf.h).  The fixtures make S singular EXACTLY -- in double, in the LU of every kernel
  and of the oracle (a zero first pivot), and in the long-double reference (det == 0): the robot's heading has zero
  variance (row 2 of P is zero) and so has the angle of a "singular" landmark (its row a is zero); a line whose R has
  R00 = R01 = 0 then gives S00 = S01 = 0 with that landmark, with no rounding anywhere.  Zero odometry keeps row 2 zero
  (Q = 0), and a match keeps both rows zero (their gain rows are exactly zero), so a singular pair stays singular in
  the later lines of a scan and in later scans.  Appended landmarks of such lines are singular too.
* More unmatched lines than free slots (SURVEY Q4): the first ones in line order are appended, the rest dropped, and
  the scan reports EKF_ECAPACITY, which takes precedence over EKF_ESINGULAR.

Every run is checked against tests/hp_reference.py: associations, line counts and status codes identical, y, the pose
and P componentwise within the reference's own bound C u mag, and zero outside the live part of the capacity layout.
tests/test_exceptional_reference.py checks the fixtures on the CPU.  The library runs in subprocesses, so that
environment knobs, the `exact` build and the mutants of section "mutants" meet the same reference run.
"""
import functools
import json
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import hp_reference as hp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TESTS = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(ROOT, "slam_ros_b200", "csrc")
FULL_MAX = 1100                      # compare every element up to this live size; sampled tiles above
SA, SR = 2e-3, 5e-3
R_REG = (SA * SA, 0.0, 0.0, SR * SR)
R_SING = (0.0, 0.0, 0.0, SR * SR)    # R00 = R01 = 0: singular S with a landmark whose angle has zero variance
R_RANK1 = (2.0 ** -18, 2.0 ** -19, 2.0 ** -19, 2.0 ** -20)   # exactly rank 1: S = R with a landmark of zero variance
NOISE = 0.01                         # line noise in units of (SA, SR)
U0 = (0.0, 0.0, 0.0)                 # zero odometry: Q = 0, the heading's variance stays exactly 0

# A line is (kind, landmark, singular R): "m" observes world landmark k, "u" sees a line 3 m beyond it (matches nothing).
M = lambda k, s=False: ("m", k, s)
N = lambda k, s=False: ("u", k, s)

# ---- single-filter cases: uploaded state, landmarks `sing` singular, scans of line specs ------------------------------
SING_SCANS = [
    # a singular landmark (1) before the true match (2); a line whose only candidate is singular (appended); a regular
    # line matching the singular landmark 4 (R00 > 0: regular); a singular pair in a later line after matches
    [M(2, True), M(1, True), M(4), M(6, True)],
    [M(0), M(3), M(5)],                                  # the next clean scan reports EKF_OK
    [M(1), M(8, True), M(9, True)],                      # singular pair (4) in later lines of a scan whose first matched
    [M(9)],
]
CAP_SCANS = [
    [M(0), N(3), N(5), M(2), N(7), N(8)],                # 4 unmatched, 3 free: the last one is dropped
    [N(1), M(4), N(2), N(6), N(9), N(0)],                # 5 unmatched, 0 free: all dropped
    [M(5)],                                              # clean
]
BOTH_SCANS = [
    [M(5, True), N(1), N(3)],                            # singular pair and one line too many: EKF_ECAPACITY
    [M(6, True)],                                        # EKF_ESINGULAR
    [M(7)],                                              # clean
]
PAST_SCANS = [
    [M(0, True)],                                        # the winner (0) comes before the singular landmarks: EKF_OK
    [M(3, True), M(5)],                                  # singular pair (1) before the winner 3
    [M(0), M(2, True)],                                  # landmark 0 matched in line 0: 1 comes first for line 1
]
RANK1_SCANS = [
    # R = [[2^-18, 2^-19], [2^-19, 2^-20]] (rank 1) with a landmark whose rows, and the robot's, are zero: S = R,
    # singular with S00 > 0
    [M(2, "r"), M(0, "r")],                              # 1 skipped before 2; 1 and 4 lie past the winner 0
    [M(3)],                                              # clean
    [M(5, "r"), M(1, "r")],                              # line 1 matches nothing: appended
]
ALL_SING_SCANS = [
    [M(0, True), M(2, True), M(3, True), M(5, True)],    # every pair singular: every line appended
    [M(1, True), M(4, True), N(0, True)],                # the appended landmarks are singular too
    [M(2)],                                              # a regular R: regular pairs
]


def _chunk_scan(n_match, n_new):
    return [M(10 + i, i % 2 == 1) for i in range(n_match)] + [N(i) for i in range(n_new)]


CASES = {
    "sing_small": dict(L=12, cap=20, headroom=0, sing=(1, 4), scans=SING_SCANS),
    "sing_past": dict(L=12, cap=20, headroom=0, sing=(1, 4), scans=PAST_SCANS),
    # the robot block and the rows of landmarks 1 and 4 are zero
    "rank1": dict(L=12, cap=20, headroom=0, sing=(1, 4), zero_robot=True, scans=RANK1_SCANS),
    "all_sing": dict(L=6, cap=20, headroom=0, sing=tuple(range(6)), scans=ALL_SING_SCANS),
    "cap_small": dict(L=10, cap=13, headroom=0, sing=(), scans=CAP_SCANS),
    "cap_reset": dict(L=10, cap=13, headroom=2, sing=(), scans=CAP_SCANS),
    "both_small": dict(L=10, cap=11, headroom=0, sing=(2,), scans=BOTH_SCANS),
    # the overlapped two-stream path: n = 3 + 2 cap >= 6000
    "sing_big": dict(L=2999, cap=3010, headroom=0, sing=(1, 4), scans=SING_SCANS),
    "past_big": dict(L=2999, cap=3010, headroom=0, sing=(1, 4), scans=PAST_SCANS),
    "cap_big": dict(L=3000, cap=3003, headroom=0, sing=(), scans=CAP_SCANS),
    "cap_big_reset": dict(L=3000, cap=3003, headroom=1, sing=(), scans=CAP_SCANS),
    # chunked scans (40 lines: chunks of 16, 16, 8): the first line that does not fit falls in the second chunk (line
    # 30, 10 lines too many) or in the last one (line 37, 3 too many); every other matched line meets the singular
    # landmarks 1 and 4 first
    "chunk_cap2": dict(L=3000, cap=3020, headroom=0, sing=(1, 4), scans=[_chunk_scan(10, 30), [M(3)]]),
    "chunk_cap3": dict(L=3000, cap=3017, headroom=0, sing=(1, 4), scans=[_chunk_scan(20, 20), [M(3)]]),
}


def _world_lines(world, pose, specs, rng):
    """z (m, 2), R (m, 4) for line specs seen from `pose`, with noise NOISE x (SA, SR)."""
    z = np.empty((len(specs), 2)); R = np.empty((len(specs), 4))
    x, yy, th = pose
    for i, (kind, k, s) in enumerate(specs):
        a, r = world[k]
        if kind == "u":
            r = r + 3.0
        z[i, 0] = np.mod(a - th + np.pi, 2 * np.pi) - np.pi
        z[i, 1] = r - (x * np.cos(a) + yy * np.sin(a))
        z[i] += rng.standard_normal(2) * np.array([SA, SR]) * NOISE
        R[i] = R_RANK1 if s == "r" else (R_SING if s else R_REG)
    return z, R


@functools.lru_cache(maxsize=None)
def case_inputs(name):
    """Start state and scans, deterministic in the case name.  P is an SPD spread state with row and column 2 (the
    heading) and the angle rows of the singular landmarks set to zero (a PSD matrix)."""
    c = CASES[name]
    seed = sum(map(ord, name.split("_")[0])) + 7
    y, P, world = hp.spread_state(c["L"], c["cap"], seed, decades=(-2.5, -1.5))
    for r in ((0, 1, 2) if c.get("zero_robot") else (2,)):
        P[r, :] = 0.0; P[:, r] = 0.0
    for j in c["sing"]:
        for r in ((3 + 2 * j, 4 + 2 * j) if c.get("zero_robot") else (3 + 2 * j,)):
            P[r, :] = 0.0; P[:, r] = 0.0
    rng = np.random.default_rng(seed)
    pose = tuple(y[:3])
    scans = [(np.array(U0),) + _world_lines(world, pose, specs, rng) for specs in c["scans"]]
    return dict(c, y=y, P=P, world=world, inputs=scans)


def blocks_for(nl, seed=0):
    """(r0, c0, nr, nc) blocks compared at live size nl."""
    if nl <= FULL_MAX:
        return [(0, 0, nl, nl)]
    t = 64 * ((nl - 1) // 64)
    out = [(0, 0, 3, nl), (t, 0, nl - t, nl), (0, t, nl, nl - t), (0, 0, 64, 64)]
    rng = np.random.default_rng(seed)
    for _ in range(8):
        r0, c0 = (int(v) * 64 for v in rng.integers(0, (nl - 1) // 64 + 1, 2))
        out.append((r0, c0, min(64, nl - r0), min(64, nl - c0)))
    return out


# ---- reference side -------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def reference(name):
    c = case_inputs(name)
    f = hp.HPFilter(c["cap"], reset_headroom=c["headroom"])
    f.upload(c["y"], c["P"], c["L"])
    out = []
    for s, (u, z, R) in enumerate(c["inputs"]):
        st, j = f.scan(u, z, R)
        r = dict(st=st, j=j, L=f.L, pose=(f.pose.copy(), f.mpose.copy()), y=(f.y[:f.nl].copy(), f.my[:f.nl].copy()),
                 C=f.C)
        if s == len(c["inputs"]) - 1:
            vals, mags = [], []
            for (r0, c0, nr, nc) in blocks_for(f.nl, s):
                v, m_ = f.block(np.arange(r0, r0 + nr), np.arange(c0, c0 + nc))
                vals.append(v.ravel()); mags.append(m_.ravel())
            r["P"] = (np.concatenate(vals), np.concatenate(mags))
        out.append(r)
    assert f.min_margin >= 1e-6, "%s: a gate decision within 1e-6 of the threshold (%g)" % (name, f.min_margin)
    return out


# ---- device side (runs in a subprocess) -----------------------------------------------------------------------------
def device_run(names, out_path, path="scan", flags=0):
    """path: "scan" (ekf_scan), "stepwise" (predict, associate, update / add_line, end_scan), "device" (ekf_scan_device,
    status from ekf_get_state's sticky word after each scan)."""
    from slam_ros_b200 import EkfFilter
    res = {}
    for name in names:
        c = case_inputs(name)
        f = EkfFilter(capacity_lines=c["cap"], reset_headroom=c["headroom"], flags=flags)
        f.upload(c["y"], c["P"], c["L"])
        if path == "device":
            import torch
            dev_in = [tuple(torch.tensor(np.ascontiguousarray(a), device="cuda") for a in inp) for inp in c["inputs"]]
            torch.cuda.synchronize()
        for s, (u, z, R) in enumerate(c["inputs"]):
            m = z.shape[0]
            if path == "stepwise":
                f.predict(u)
                j = np.full(m, -1, np.int32)
                for i in range(m):
                    j[i], _ = f.associate(z[i], R[i])
                    if j[i] >= 0:
                        f.update(j[i], z[i], R[i])
                    else:
                        f.add_line(z[i], R[i])
                rc, pose = f.end_scan(m)
            elif path == "device":
                import torch
                du, dz, dR = dev_in[s]
                dj = torch.full((m,), -7, dtype=torch.int32, device="cuda")
                f.scan_device(du.data_ptr(), m, dz.data_ptr(), dR.data_ptr(), dj.data_ptr())
                pose, L, rc = f.state()
                j = dj.cpu().numpy()
            else:
                rc, j, pose = f.scan(u, z, R)
            k = "%s/%d/" % (name, s)
            res[k + "st"] = np.array(rc); res[k + "j"] = j; res[k + "pose"] = pose
            res[k + "L"] = np.array(f.lines); res[k + "y"] = f.download_y()
            if s == len(c["inputs"]) - 1:
                nl = 3 + 2 * f.lines
                res[k + "P"] = np.concatenate([f.download_block(*b).ravel() for b in blocks_for(nl, s)])
                yc, Pc, Lc = f.download()
                res[k + "dead"] = np.array([bool(yc[nl:].any() or Pc[nl:].any() or Pc[:, nl:].any())])
                res[k + "after"] = np.array(f.state()[2])       # the sticky word was cleared by the scan's read
        f.close()
    np.savez(out_path, **res)


def _spawn(call, env_extra, lib=None):
    path = os.path.join("/tmp", "ekf_exceptional_%d_%s.npz" % (
        os.getpid(), abs(hash((call, json.dumps(env_extra, sort_keys=True), str(lib))))))
    code = "import sys; sys.path[:0] = [%r, %r]\nimport test_gpu_exceptional as t\n%s\n" % (ROOT, TESTS, call % path)
    env = dict(os.environ)
    for k in ("EKF_LINE_LOOP", "EKF_LIB", "EKF_BATCH_NS", "EKF_CHUNK", "EKF_CHUNK_ABOVE"):
        env.pop(k, None)
    env.update(env_extra)
    if lib:
        env["EKF_LIB"] = lib
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=1200, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    res = dict(np.load(path))
    os.remove(path)
    return res


def compare(dev, names, label, raise_=True):
    """Every check of the cases.  Returns (worst err / (C u mag) per quantity, failures)."""
    worst = {"y": 0.0, "pose": 0.0, "P": 0.0}
    fails = []
    for name in names:
        for s, r in enumerate(reference(name)):
            k = "%s/%d/" % (name, s)
            what = "%s %s" % (label, k)
            if not np.array_equal(dev[k + "j"], r["j"]):
                fails.append("%s associations %s vs reference %s" % (what, dev[k + "j"], r["j"]))
            if int(dev[k + "st"]) != r["st"]:
                fails.append("%s status %d vs reference %d" % (what, int(dev[k + "st"]), r["st"]))
            if int(dev[k + "L"]) != r["L"]:
                fails.append("%s line count %d vs reference %d" % (what, int(dev[k + "L"]), r["L"]))
                continue
            for q in ("pose", "y", "P"):
                if q not in r:
                    continue
                v, m_ = r[q]
                if dev[k + q].shape != v.shape:
                    fails.append("%s %s shape %s vs %s" % (what, q, dev[k + q].shape, v.shape))
                    continue
                w = hp.worst_ratio(dev[k + q], v, m_)
                worst[q] = max(worst[q], w / r["C"])
                if w > r["C"]:
                    fails.append("%s %s: worst |x - ref| / (u mag) = %.3g > C = %d" % (what, q, w, r["C"]))
            if k + "dead" in dev and bool(dev[k + "dead"][0]):
                fails.append("%s nonzero entries outside the live part" % what)
            if k + "after" in dev and int(dev[k + "after"]) != 0:
                fails.append("%s sticky status %d after the scan's own read" % (what, int(dev[k + "after"])))
    if raise_:
        assert not fails, "%d failures, first: %s" % (len(fails), fails[:4])
    print("exceptional %-12s worst err/(C u mag): y %.2e  pose %.2e  P %.2e" % (label, worst["y"], worst["pose"], worst["P"]))
    return worst, fails


# path -> (environment, flags, ekf entry, cases): one singular and one capacity case per path
PATHS = {
    "stepwise": ({}, 0, "stepwise", ["sing_small", "sing_past", "rank1", "cap_small"]),
    "fused": ({}, 0, "scan", ["sing_small", "sing_past", "rank1", "all_sing", "cap_small", "cap_reset", "both_small"]),
    "line_loop1": ({"EKF_LINE_LOOP": "1"}, 0, "scan", ["sing_small", "sing_past", "rank1", "cap_small"]),
    "per_line": ({}, 4, "scan", ["sing_small", "sing_past", "rank1", "both_small"]),
    "eager": ({}, 1, "scan", ["all_sing", "sing_past", "rank1", "cap_reset"]),
    "overlap": ({}, 0, "scan", ["sing_big", "past_big", "cap_big", "cap_big_reset"]),
    "no_overlap": ({}, 8, "scan", ["sing_big", "past_big", "cap_big"]),
    "chunked": ({}, 0, "scan", ["chunk_cap2", "chunk_cap3"]),
    "device": ({}, 0, "device", ["sing_small", "sing_past", "both_small", "cap_big"]),
    "exact_build": ({"EKF_LIB": "exact"}, 0, "scan", ["sing_small", "sing_past", "cap_small"]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PATHS))
def test_single_filter_exceptional(libekf, path):
    env, flags, entry, names = PATHS[path]
    if env.get("EKF_LIB") == "exact":
        from slam_ros_b200 import build as b
        env = dict(env, EKF_LIB=b.build_variant("exact"))
    dev = _spawn("t.device_run(%r, %%r, path=%r, flags=%d)" % (names, entry, flags), env)
    compare(dev, names, path)


# ---- batch filters --------------------------------------------------------------------------------------------------
# Seeded from the empty map: scan 0 appends L0 landmarks per filter from the pose (0, 0, 0), whose heading has zero
# variance.  A landmark appended with R00 = R01 = 0 has an angle of zero variance: singular with a line of R_SING.
# "small": every landmark in one round of the pre-test and of the full gates.  "rounds": 70 landmarks, so that the
# singular pairs before a winner fill whole rounds of full gates (filter 0), and singular pairs lie rounds past a
# winner, where first fit never gates them (filter 1).
BATCHES = {
    "small": dict(cap=14, L0=12, sing=[(1, 4), (3,), (), tuple(range(12))], plan=[   # per scan: each filter's lines
        [[M(2, True), M(1, True), M(4), M(6, True)],    # f0 singular; f1 clean; f2 one line too many; f3 both
         [M(0), M(3), M(5), M(7)],
         [N(0), N(3), N(5), M(2)],
         [M(0, True), M(2, True), N(3, True), M(5, True)]],
        [[M(0), M(3), M(5)], [M(6, True), M(8), M(9)], [M(1), M(4), M(6)], [M(1), M(7), M(8)]],   # f1 singular only
        # clean: f0's first line matches landmark 0, its singular pairs (1, 4) lie past the winner in the same round
        [[M(0, True), M(8)], [M(0), M(2)], [M(3), M(5)], [M(9), M(10)]],
        [[M(9), M(10), M(11)], [M(4), M(5), M(6)], [N(7), N(8), N(9)], [M(2), M(3), M(4)]],      # f2 3 too many
    ]),
    "rounds": dict(cap=80, L0=70, sing=[tuple(range(40)), tuple(range(40, 70))], plan=[
        [[M(50, True), M(60, True)], [M(5, True), M(6, True)]],     # f0: 40 singular pairs first; f1: all past
        [[M(45), M(10)], [M(4, True), M(50)]],                      # clean (f1 line 0: singular pairs past 4)
        [[M(45, True)], [M(45)]],                                   # f0 singular; f1 regular pairs only
    ]),
}
# the batch's own knobs: the on-chip triangle's width (3: every appended column goes to HBM) and full gates
B_VARIANTS = {"default": ({}, 0, 0), "full_gates": ({}, 16, 0), "ns3": ({"EKF_BATCH_NS": "3"}, 0, 0),
              "pipelined": ({}, 0, 1)}


@functools.lru_cache(maxsize=None)
def batch_inputs(kind):
    c = BATCHES[kind]
    B = len(c["sing"])
    rng = np.random.default_rng(2024)
    worlds = [hp.spread_state(c["L0"], c["L0"], 900 + f)[2] for f in range(B)]
    scans = []
    z = np.array([w.copy() for w in worlds])
    R = np.array([[R_SING if (k in c["sing"][f]) else R_REG for k in range(c["L0"])] for f in range(B)])
    scans.append((np.zeros((B, 3)), z, R))
    for plan in c["plan"]:
        zz, RR = zip(*[_world_lines(worlds[f], (0.0, 0.0, 0.0), plan[f], rng) for f in range(B)])
        scans.append((np.zeros((B, 3)), np.array(zz), np.array(RR)))
    return scans


def batch_status(sts):
    """ekf_batch_collect's aggregation: EKF_ECAPACITY if any filter overflowed, else EKF_ESINGULAR if any met a
    singular pair."""
    return 2 if 2 in sts else (3 if 3 in sts else 0)


@functools.lru_cache(maxsize=None)
def batch_reference(kind, headroom):
    c = BATCHES[kind]
    filters = [hp.HPFilter(c["cap"], reset_headroom=headroom) for _ in c["sing"]]
    out = []
    for (u, z, R) in batch_inputs(kind):
        res = [f.scan(u[i], z[i], R[i]) for i, f in enumerate(filters)]
        out.append(dict(st=batch_status([r[0] for r in res]), fst=[r[0] for r in res], j=np.stack([r[1] for r in res]),
                        pose=[(f.pose.copy(), f.mpose.copy(), f.C) for f in filters]))
    states = [(f.L, f.live(), f.C) for f in filters]
    assert min(f.min_margin for f in filters) >= 1e-6
    return out, states


def batch_device(out_path, kind, headroom, flags=0, pipelined=0):
    from slam_ros_b200 import EkfBatch
    c = BATCHES[kind]
    scans = batch_inputs(kind)
    bt = EkfBatch(len(c["sing"]), capacity_lines=c["cap"], reset_headroom=headroom, flags=flags)
    res = {}
    if pipelined:                     # step s + 1 is submitted before step s is collected
        bt.submit(*scans[0])
        for s in range(len(scans)):
            if s + 1 < len(scans):
                bt.submit(*scans[s + 1])
            rc, j, pose = bt.collect()
            res["%d/st" % s] = np.array(rc); res["%d/j" % s] = j; res["%d/pose" % s] = pose
    else:
        for s, (u, z, R) in enumerate(scans):
            rc, j, pose = bt.scan(u, z, R)
            res["%d/st" % s] = np.array(rc); res["%d/j" % s] = j; res["%d/pose" % s] = pose
    for f in range(len(c["sing"])):
        y, P, L, pose = bt.download(f)
        res["f%d/y" % f] = y; res["f%d/P" % f] = P; res["f%d/L" % f] = np.array(L)
    bt.close()
    np.savez(out_path, **res)


def batch_compare(dev, kind, headroom, label, raise_=True):
    ref, states = batch_reference(kind, headroom)
    fails = []
    worst = 0.0
    for s, r in enumerate(ref):
        if not np.array_equal(dev["%d/j" % s], r["j"]):
            fails.append("%s scan %d: associations %s vs reference %s" % (label, s, dev["%d/j" % s], r["j"]))
        if int(dev["%d/st" % s]) != r["st"]:
            fails.append("%s scan %d: status %d vs reference %d (filters %s)" % (label, s, int(dev["%d/st" % s]), r["st"], r["fst"]))
        for f, (pv, pm, C) in enumerate(r["pose"]):
            if hp.worst_ratio(dev["%d/pose" % s][f], pv, pm) > C:
                fails.append("%s scan %d filter %d: pose" % (label, s, f))
    for f, (L, (yv, ym, Pv, Pm), C) in enumerate(states):
        if int(dev["f%d/L" % f]) != L:
            fails.append("%s filter %d: line count %d vs reference %d" % (label, f, int(dev["f%d/L" % f]), L))
            continue
        nl = 3 + 2 * L
        for q, d, v, m_ in (("y", dev["f%d/y" % f][:nl], yv, ym), ("P", dev["f%d/P" % f][:nl, :nl], Pv, Pm)):
            w = hp.worst_ratio(d, v, m_)
            worst = max(worst, w / C)
            if w > C:
                fails.append("%s filter %d %s: worst |x - ref| / (u mag) = %.3g > C = %d" % (label, f, q, w, C))
        if dev["f%d/y" % f][nl:].any() or dev["f%d/P" % f][nl:].any() or dev["f%d/P" % f][:, nl:].any():
            fails.append("%s filter %d: nonzero entries outside the live part" % (label, f))
    if raise_:
        assert not fails, "%d failures, first: %s" % (len(fails), fails[:4])
    print("exceptional batch %-6s %-10s headroom %d worst P err/(C u mag) %.2e" % (kind, label, headroom, worst))
    return fails


@pytest.mark.gpu
@pytest.mark.parametrize("kind,variant,headroom", [("small", v, h) for v in B_VARIANTS for h in (0, 1)] +
                         [("rounds", "default", 0), ("rounds", "full_gates", 0)])
def test_batch_exceptional(libekf, kind, variant, headroom):
    env, flags, pipelined = B_VARIANTS[variant]
    dev = _spawn("t.batch_device(%%r, %r, %d, flags=%d, pipelined=%d)" % (kind, headroom, flags, pipelined), env)
    batch_compare(dev, kind, headroom, variant)


# ---- the Python mirror passes both codes through ---------------------------------------------------------------------
@pytest.mark.gpu
def test_robot_mirror_passes_both_codes(libekf):
    from slam_ros_b200.robot import Robot, Line
    from slam_ros_b200.ekf import EKF_ECAPACITY, EKF_ESINGULAR, EKF_OK
    rb = Robot(linesize=3, reset_headroom=0)
    # a fresh filter's heading has zero variance: lines with R00 = R01 = 0 append landmarks whose angle has none either
    first = [Line(0.0, 2.0, R_SING), Line(1.0, 3.0, R_REG)]
    assert rb.localize(first, encoder=(0.0, 0.0, 0.0)) == EKF_OK and rb.savedLineCount == 2
    # line 0: singular with landmark 0, no other candidate: appended; line 1 matches landmark 1; line 2 does not fit
    second = [Line(0.0, 2.0, R_SING), Line(1.0, 3.0, R_REG), Line(-1.0, 4.0, R_REG)]
    assert rb.localize(second, encoder=(0.0, 0.0, 0.0)) == EKF_ECAPACITY and rb.savedLineCount == 3
    assert list(rb.last_matches) == [-1, 1, -1]
    # singular with landmark 0, then a match with landmark 1
    third = [Line(1.0, 3.0, R_SING)]
    assert rb.localize(third, encoder=(0.0, 0.0, 0.0)) == EKF_ESINGULAR and list(rb.last_matches) == [1]


@pytest.mark.gpu
def test_cpp_robot_passes_both_codes(libekf, tmp_path):
    from slam_ros_b200.ekf import library_path
    exe = str(tmp_path / "status_main")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([cxx, "-std=c++11", "-O2", "-I", os.path.join(ROOT, "include"),
                           os.path.join(TESTS, "cpp", "status_main.cpp"), library_path(),
                           "-Wl,-rpath," + os.path.dirname(library_path()), "-o", exe])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "status_main OK" in out.stdout, out.stdout + out.stderr


# ---- mutants ----------------------------------------------------------------------------------------------------------
# (file, anchor, replacement, what it breaks, test that must catch it).  Each changes values only: no index, size, loop
# bound, barrier or stream order, so none can fault or hang.
MUTANTS = {
    "a": ("ekf_kernels.cu",
          "/* reported by k_end_scan_a if below the winner */\n        else if (!gate_rejects_d2(G.d2, g.gate_d2max)) { cand = j;",
          "/* reported by k_end_scan_a if below the winner */\n        if (!gate_rejects_d2(G.d2, g.gate_d2max)) { cand = j;",
          "the two-barrier line loop (EKF_LINE_LOOP=1) ends a line's first fit at a singular pair (S^-1 = 0, d2 = 0)",
          ("single", "line_loop1")),
    "b": ("ekf_batch.cu", "(g.full_gates || !(S00 > 0.0) || !(v * v > gate2x4 * S00))",
          "(g.full_gates || !(v * v > gate2x4 * S00))",
          "the batch pre-test discards landmarks with S00 == 0", ("batch", "default")),
    "c": ("ekf_kernels.cu", "const int n_add = min(ne, g.cap - L);", "const int n_add = min(ne, max(g.cap - L - 1, 0));",
          "the single filter's capacity test is off by one", ("single", "fused")),
    "d": ("ekf_batch.cu", "if (sing < best) atomicOr(&s_sticky, EKF_STICKY_SINGULAR);",
          "if (sing < best) atomicOr(&s_sticky, 0);",
          "the batch never sets the singular sticky bit", ("batch", "full_gates")),
    "e": ("ekf_kernels.cu", "skipped |= b.jsing[i] < b.jbest[i];", "skipped |= b.jsing[i] != EKF_NO_MATCH;",
          "the single filter reports singular pairs past a line's winner", ("single", "fused")),
}


def test_mutant_anchors_occur_exactly_once():
    """A refactor that moves or rewrites one of the guarded lines breaks the mutant list here, not silently."""
    for key, (fname, anchor, repl, what, (kind, variant)) in MUTANTS.items():
        with open(os.path.join(CSRC, fname)) as fh:
            n = fh.read().count(anchor)
        assert n == 1, "%s: anchor %r occurs %d times in %s" % (key, anchor, n, fname)
        assert variant in (PATHS if kind == "single" else B_VARIANTS)


def build_mutant(key, workdir):
    """Copies slam_ros_b200/csrc and include (same relative layout), applies mutant `key`, starts nvcc.  Returns
    (process, library path)."""
    from slam_ros_b200 import build as b
    fname, anchor, repl = MUTANTS[key][:3]
    src = os.path.join(workdir, "slam_ros_b200", "csrc")
    shutil.copytree(CSRC, src)
    shutil.copytree(os.path.join(ROOT, "include"), os.path.join(workdir, "include"))
    path = os.path.join(src, fname)
    with open(path) as fh:
        text = fh.read()
    assert text.count(anchor) == 1, (key, anchor)
    with open(path, "w") as fh:
        fh.write(text.replace(anchor, repl))
    out = os.path.join(workdir, "libekfcuda_%s.so" % key)
    cmd = [b.nvcc_path()] + b.NVCC_FLAGS + [os.path.join(src, s) for s in b.SOURCES] + ["-o", out, "-ldl"]
    return subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True), out


@pytest.fixture(scope="module")
def mutant_libs(tmp_path_factory):
    procs = {k: build_mutant(k, str(tmp_path_factory.mktemp("exc_mutant_" + k))) for k in MUTANTS}
    libs = {}
    for k, (p, out) in procs.items():
        log, _ = p.communicate(timeout=1800)
        assert p.returncode == 0, "%s: nvcc failed\n%s" % (k, log[-3000:])
        libs[k] = out
    return libs


@pytest.mark.gpu
@pytest.mark.parametrize("key", list(MUTANTS))
def test_each_exceptional_branch_is_guarded(libekf, mutant_libs, key):
    fname, anchor, repl, what, (kind, variant) = MUTANTS[key]
    if kind == "single":
        env, flags, entry, names = PATHS[variant]
        dev = _spawn("t.device_run(%r, %%r, path=%r, flags=%d)" % (names, entry, flags), env, mutant_libs[key])
        worst, fails = compare(dev, names, "mutant " + key, raise_=False)
    else:
        env, flags, pipelined = B_VARIANTS[variant]
        dev = _spawn("t.batch_device(%%r, 'small', 0, flags=%d, pipelined=%d)" % (flags, pipelined), env,
                     mutant_libs[key])
        fails = batch_compare(dev, "small", 0, "mutant " + key, raise_=False)
    print("mutant %s (%s): %d failures, first: %s" % (key, what, len(fails), fails[0] if fails else "-"))
    assert fails, "mutant %s (%s) passes: %s is not guarded" % (key, repl, what)
