"""The overlapped two-stream pipeline and its sweep groups against the extended-precision reference, element by element.

`test_gpu_componentwise.py` reads y after every scan, and every download drains the pipeline: its scans always start with
no sweep in flight and a group of one.  Here long sequences run on the overlapped path with no observer of P or y
between scans, so that a scan's line loop corrects its column reads against the previous group's still-pending terms
while that group's sweep is in flight, and two or more scans share one sweep (DESIGN section 5).  Between scans only hot
storage is read: associations, line count, pose and the 3x3 robot covariance.  At the end y and P are compared with
hp.HPFilter run over the same inputs, |x - ref| <= C u mag(x), C from the reference's operation count.

Every case also asserts that it exercised what it is meant to: the sweep launches and the terms they folded are those of
the intended grouping (profile_read), ghosts appended in the first scan of a group are matched in the next, the reset
falls inside a group, the deepest line corrects against FL_MAXP - 1 = 127 pending terms.

test_each_pipeline_invariant_is_guarded rebuilds the library with one of the group invariants removed and requires the
comparison to fail.  The anchors of those mutants are checked on the CPU (test_mutant_anchors_occur_exactly_once).
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
FULL_MAX = 1100             # compare every element up to this live size; rows, tiles and landmark rows above
U_STEP = (0.02, 0.0, 0.01)
OVERLAP_MIN_N = 6000        # kOverlapMinN (ekf_api.cu): below this state dimension scans do not overlap


def _ragged(ms):
    """A plan of the given line counts: from 3 lines on, one ghost per scan, re-observed by the next scan of 4 or more."""
    plan, prev_new = [], 0
    for m in ms:
        if m < 3:
            plan.append((0, m, 0)); prev_new = 0
            continue
        again = 1 if (prev_new and m >= 4) else 0
        plan.append((again, m - again - 1, 1)); prev_new = 1
    return plan


RAGGED_MS = [8, 3, 5, 12, 1, 16, 0, 8, 40, 5, 3, 8, 12, 12, 1, 1, 1, 8]

# name -> L0, capacity (= 126 mod 128: n = 255 mod 256), reset headroom, plan, scans on the device-resident path,
# warm-up on a larger map first, environment the case needs.
# A plan entry (again, true, new): `again` lines appended by the previous scan seen again, `true` lines of the
# uploaded map's landmarks, `new` ghosts (a landmark's line 3 m further out: matches nothing, is appended).
CASES = {
    # a. groups of two, m = 8: ghosts appended by the first scan of a group are matched by the second; the third group's
    #    first scan takes nl from 6013 to 6019 across the tile boundary at 6016; ends at nl = 6017 = 1 (mod 64)
    "groups_nl1": dict(L=3000, cap=3070, headroom=0, plan=[(0, 5, 3), (3, 5, 0)] + [(0, 6, 2), (2, 6, 0)] * 2),
    #    ... and at nl = 6015 = 63 (mod 64)
    "groups_nl63": dict(L=3000, cap=3070, headroom=0, plan=[(0, 6, 2), (2, 6, 0)] * 3),
    # b. ragged line counts at capacity 10 366: groups close on the budget, on a chunked scan (40 lines), on an empty
    #    scan and on a change of line-loop class (m > 8 takes 21 SMs at this capacity, m <= 8 takes 20)
    "ragged": dict(L=3000, cap=10366, headroom=0, plan=_ragged(RAGGED_MS)),
    # c. map reset in the first scan of a group (L > capacity - headroom after scan 6), device-resident scans; the
    #    rebuilt map is re-observed by the scans after it
    "reset": dict(L=3300, cap=3326, headroom=10, device=True,
                  plan=[(0, 6, 2)] * 6 + [(0, 3, 5), (0, 8, 0), (4, 4, 0), (4, 4, 0), (4, 4, 0), (4, 4, 0)]),
    # d. eight scans per sweep: the last line of the second group corrects against 64 + 63 pending terms; the third
    #    group holds an odd number of terms and is still open when the sequence ends
    "deep": dict(L=3000, cap=3070, headroom=0, env={"EKF_SWEEP_GROUP": "64"},
                 plan=[(0, 8, 0)] * 16 + [(0, 7, 1), (1, 7, 0), (0, 8, 0)]),
    # e. as a, after a warm-up on a map of L0 + 40 landmarks that leaves stale terms in both halves of the slot ring at
    #    the rows this sequence appends (ekf_upload does not clear the slots)
    "stale": dict(L=3000, cap=3070, headroom=0, warm=True, plan=[(0, 6, 2), (2, 6, 0)] * 3),
    # c on a map the CPU oracle handles in seconds (tests/test_hp_reference.py): the same plan, reset in scan 6
    "reset_small": dict(L=360, cap=382, headroom=10,
                        plan=[(0, 6, 2)] * 6 + [(0, 3, 5), (0, 8, 0), (4, 4, 0), (4, 4, 0), (4, 4, 0), (4, 4, 0)]),
}
WARM_SCANS = 6


def case_inputs(name):
    """Start state and the scans' inputs, deterministic in the case name."""
    c = CASES[name]
    L0, cap, headroom = c["L"], c["cap"], c["headroom"]
    seed = sum(map(ord, name))
    rng = np.random.default_rng(seed)
    y, P, world0 = hp.spread_state(L0, cap, seed)
    world = [tuple(w) for w in world0]
    in_map = list(range(L0))          # world line of every landmark, as the plan intends the map to evolve
    placed = {}                       # world line -> the line an appended landmark holds (see below)
    pose = tuple(y[:3])
    prev_new, scans = [], []
    for again, t, new in c["plan"]:
        pose = hp.predicted_pose(pose, U_STEP)
        ids = list(prev_new[:again]) + [int(i) for i in rng.choice(L0, t, replace=False)]
        for _ in range(new):
            src = int(rng.integers(L0))
            world.append((world[src][0], world[src][1] + 3.0))
            ids.append(len(world) - 1)
        if ids:
            z, R = hp.lines_for(np.array([placed.get(i, world[i]) for i in ids]), pose, range(len(ids)), rng)
        else:
            z, R = np.zeros((0, 2)), np.zeros((0, 4))
        known = set(in_map)
        appended = [i for i in ids if i not in known]
        for k, i in enumerate(ids):
            if i not in known:
                # Robot.cpp:792 converts the range with the angle in the robot frame: an appended landmark sits where
                # that puts it, and the lines that re-observe it are generated from there (so that they match it)
                a = z[k, 0] + pose[2]
                placed[i] = (float(np.mod(a + np.pi, 2 * np.pi) - np.pi),
                             z[k, 1] + pose[0] * np.cos(z[k, 0]) + pose[1] * np.sin(z[k, 0]))
        in_map += appended
        prev_new = appended
        if len(in_map) > cap - headroom:
            in_map, prev_new, placed = [], [], {}
        scans.append((np.array(U_STEP), z, R))
    out = dict(L=L0, cap=cap, headroom=headroom, y=y, P=P, scans=scans)
    if c.get("warm"):
        wy, wP, wworld = hp.spread_state(L0 + 40, cap, seed + 1)
        wpose, wscans = tuple(wy[:3]), []
        for _ in range(WARM_SCANS):
            wpose = hp.predicted_pose(wpose, U_STEP)
            z, R = hp.lines_for(wworld, wpose, rng.choice(L0 + 40, 8, replace=False), rng)
            wscans.append((np.array(U_STEP), z, R))
        out["warm"] = (wy, wP, L0 + 40, wscans)
    return out


# ---- the intended grouping (the host rules of DESIGN section 5) -------------------------------------------------------
def knobs(env, max_batch=64):
    """The host's sizing of the slot ring and the group budget (ekf_api.cu, create_common) for ekf_config.max_batch:
    group = 64 from max_batch = 64 on, else min(max_batch / 2, 32); slots (rows of Kp / KSp) = max(max_batch, 2 group);
    then group capped at 2 x ekf_sweep_terms_per_pass(shape, 64), which is min(32, EKF_SWEEP_MAXC) for the sweep shapes
    the variants use (0, 10, 11); budget = min(EKF_SWEEP_GROUP or 16, group); chunks of min(16, group) lines above 32.
    Below max_batch = 16 nothing overlaps.  If that sizing changes, update this function: the grouping assertions
    depend on it."""
    mb = max_batch if max_batch > 0 else 64
    maxc = int(env.get("EKF_SWEEP_MAXC", 32))
    maxc = maxc if maxc in (8, 16, 32) else 32
    group = 64 if mb >= 64 else min(mb // 2, 32)
    slots = max(mb, 2 * group)
    group = max(1, min(group, 2 * min(32, maxc)))   # ring half: 2 x ekf_sweep_terms_per_pass(shape 0/9/10/11, 64)
    budget = max(0, min(int(env.get("EKF_SWEEP_GROUP", 16)), group))
    return dict(group=group, slots=slots, budget=budget, chunk=min(16, group), chunk_above=32, max_batch=mb,
                overlap=mb >= 16, line_sms=int(env.get("EKF_LINE_SMS", -1)))


def line_sms(m, cap, k):
    if 1 <= k["line_sms"] <= 64:
        return k["line_sms"]
    need = (cap + 511) // 512
    return need if (m > 8 and 20 < need <= 28) else 20


def inplace_bounds(m, max_batch):
    """Term bounds of the in-place sweeps of one scan of m lines on a non-empty map: the fused line loop (max_batch <= 64)
    and the per-line kernels both fold every max_batch lines and at the end of the scan."""
    return [min(max_batch, m - l0) for l0 in range(0, m, max_batch)]


def intended_grouping(ms, cap, env, max_batch=64, halves=None):
    """(term bound of every sweep, scans of every sweep) for scans of ms lines on a map that stays on the overlapped
    path, with a sync at the end.  A scan of 0 lines, or of more than the ring half and unchunked, drains and runs in
    place: one sweep per max_batch lines.  `halves`, if a list, receives the slot-ring half of every sweep (0 or 1; None
    for an in-place sweep): the ring starts at half 0 when the filter is created and alternates at every hand-off."""
    k = knobs(env, max_batch)
    bounds, members = [], []
    cur = None                                   # [term bound, line-loop SMs, scans] of the open group
    par = [0]

    def add(bound, scans, ring=True):
        bounds.append(bound); members.append(scans)
        if halves is not None:
            halves.append(par[0] if ring else None)
        if ring:
            par[0] ^= 1

    def close():
        nonlocal cur
        if cur is not None:
            add(cur[0], cur[2]); cur = None

    for s, m in enumerate(ms):
        chunked = k["chunk"] > 0 and m > k["chunk_above"]
        if m < 1 or (m > k["group"] and not chunked):
            close()
            for b in inplace_bounds(m, k["max_batch"]):
                add(b, [s], ring=False)
            continue
        ls = line_sms(m, cap, k)
        groupable = k["budget"] > 0 and not chunked
        joins = groupable and cur is not None and cur[0] + m <= k["budget"] and ls == cur[1]
        if not joins:
            close()
        if not groupable:
            step = k["chunk"] if chunked else m
            for l0 in range(0, m, step):
                add(min(step, m - l0), [s])
            continue
        if cur is None:
            cur = [0, ls, []]
        cur[0] += m; cur[2].append(s)
        if cur[0] + m > k["budget"]:
            close()
    close()
    return bounds, members


def deepest_correction(members, J):
    """Most pending terms any matched line corrects against: the previous group's terms (its sweep is in flight) plus
    the terms its own group formed before it.  The first group after an upload has no previous group."""
    deepest, prev = 0, 0
    for gi, scans in enumerate(members):
        own = 0
        for s in scans:
            for j in J[s]:
                if j >= 0:
                    deepest = max(deepest, prev + own)
                    own += 1
        prev = own
    return deepest


def blocks_for(nl, rows, seed=0):
    """(r0, c0, nr, nc) blocks compared at live size nl; `rows`: landmarks whose full rows are compared."""
    if nl <= FULL_MAX:
        return [(0, 0, nl, nl)]
    t = 64 * ((nl - 1) // 64)
    out = [(0, 0, 3, nl), (t, 0, nl - t, nl), (0, t, nl, nl - t)]
    out += [(d, d, min(64, nl - d), min(64, nl - d)) for d in range(0, nl, 64)]
    out += [(3 + 2 * j, 0, 2, nl) for j in sorted(rows) if 3 + 2 * j + 1 < nl]
    rng = np.random.default_rng(seed)
    for _ in range(32):
        r0, c0 = (int(v) * 64 for v in rng.integers(0, (nl - 1) // 64 + 1, 2))
        out.append((r0, c0, min(64, nl - r0), min(64, nl - c0)))
    return out


# ---- reference side -----------------------------------------------------------------------------------------------
def _sym3(T):
    """The 3x3 robot block as ekf_get_robot_cov returns it: the upper triangle mirrored."""
    A = np.array(T[:, :3])
    return np.triu(A) + np.triu(A, 1).T


@functools.lru_cache(maxsize=None)
def reference(name):
    c = case_inputs(name)
    f = hp.HPFilter(c["cap"], reset_headroom=c["headroom"])
    f.upload(c["y"], c["P"], c["L"])
    per_scan, touched = [], set()
    for u, z, R in c["scans"]:
        L_before = f.L
        st, j = f.scan(u, z, R)
        reset = f.L < L_before
        if reset:
            touched = set()                      # the landmarks touched so far belong to the old map
        else:
            touched |= set(int(v) for v in j if v >= 0) | set(range(L_before, f.L))
        per_scan.append(dict(j=j, L_before=L_before, L=f.L, reset=reset,
                             pose=(f.pose.copy(), f.mpose.copy()), rcov=(_sym3(f.T), _sym3(f.mT)), C=f.C))
    assert f.min_margin >= 1e-6, "%s: a gate decision within 1e-6 of the threshold (%g)" % (name, f.min_margin)
    blocks = blocks_for(f.nl, touched, len(c["scans"]))
    vals, mags = [], []
    for r0, c0, nr, nc in blocks:
        v, m_ = f.block(np.arange(r0, r0 + nr), np.arange(c0, c0 + nc))
        vals.append(v.ravel()); mags.append(m_.ravel())
    return dict(scans=per_scan, L=f.L, y=(f.y[:f.nl].copy(), f.my[:f.nl].copy()), blocks=blocks,
                P=(np.concatenate(vals), np.concatenate(mags)), C=f.C, touched=len(touched))


# ---- device side (runs in a subprocess, with the environment under test) --------------------------------------------
def device_run(name, blocks, out_path, cfg=None):
    """cfg: further ekf_config fields (max_batch, flags) of the filter under test."""
    from slam_ros_b200 import EkfFilter
    c = case_inputs(name)
    spec = CASES[name]
    res = {}
    f = EkfFilter(capacity_lines=c["cap"], reset_headroom=c["headroom"], **(cfg or {}))
    if "warm" in c:
        wy, wP, wL, wscans = c["warm"]
        f.upload(wy, wP, wL)
        res["warm_matched"] = np.array(sum(int((f.scan(u, z, R)[1] >= 0).sum()) for u, z, R in wscans))
    f.upload(c["y"], c["P"], c["L"])
    f.profile_enable(True)
    if spec.get("device"):
        import torch
        dev = torch.device("cuda")
        S = len(c["scans"])
        mmax = max(max(z.shape[0] for _, z, _ in c["scans"]), 1)
        d_u = torch.tensor(np.stack([u for u, _, _ in c["scans"]]), device=dev)
        d_z = [torch.tensor(z, device=dev) for _, z, _ in c["scans"]]
        d_R = [torch.tensor(R, device=dev) for _, _, R in c["scans"]]
        d_j = torch.full((S, mmax), -7, dtype=torch.int32, device=dev)
        for s, (u, z, R) in enumerate(c["scans"]):
            f.scan_device(d_u[s].data_ptr(), z.shape[0], d_z[s].data_ptr(), d_R[s].data_ptr(), d_j[s].data_ptr())
        f.sync()
        J = d_j.cpu().numpy()
        for s, (u, z, R) in enumerate(c["scans"]):
            res["%d/j" % s] = J[s, :z.shape[0]]
        pose, L, _ = f.state()
        res["end/pose"] = pose; res["end/L"] = np.array(L); res["end/rcov"] = f.robot_cov()
    else:
        for s, (u, z, R) in enumerate(c["scans"]):
            rc, j, pose = f.scan(u, z, R)
            res["%d/j" % s] = j; res["%d/pose" % s] = pose
            res["%d/L" % s] = np.array(f.lines); res["%d/rcov" % s] = f.robot_cov()
        f.sync()
    prof = f.profile_read()
    f.profile_enable(False)
    res["prof"] = np.array([prof["sweeps"], prof["sweep_bytes"]])
    L = f.lines
    res["L"] = np.array(L)
    res["y"] = f.download_y()
    nl = 3 + 2 * L
    if all(r0 + nr <= nl and c0 + nc <= nl for r0, c0, nr, nc in blocks):
        res["P"] = np.concatenate([f.download_block(*b).ravel() for b in blocks])
    f.close()
    np.savez(out_path, **res)


def _spawn(name, env_extra, workdir, lib=None, cfg=None, module=None):
    """device_run(name, cfg) in a child process with the environment under test; its results go to a file in workdir.
    module: a test module to import first in the child (one that adds its own cases to CASES)."""
    ref = reference(name)
    key = json.dumps([env_extra, cfg], sort_keys=True) + str(lib)
    path = os.path.join(str(workdir), "%s_%s.npz" % (name, abs(hash(key))))
    code = ("import sys; sys.path[:0] = [%r, %r]\n%simport test_gpu_pipeline_componentwise as t\n"
            "t.device_run(%r, %r, %r, %r)\n" % (ROOT, TESTS, ("import %s\n" % module) if module else "", name,
                                                  [list(b) for b in ref["blocks"]], path, cfg))
    env = dict(os.environ)
    for k in ("EKF_SWEEP_GROUP", "EKF_SWEEP_MAXC", "EKF_SWEEP_SHAPE", "EKF_LINE_LOOP", "EKF_LINE_SMS", "EKF_FUSE_PREDICT",
              "EKF_LIB", "EKF_CHUNK", "EKF_CHUNK_ABOVE", "EKF_LINE_THREADS"):
        env.pop(k, None)
    env.update(CASES[name].get("env", {}))
    env.update(env_extra)
    if lib:
        env["EKF_LIB"] = lib
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=1200, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    res = dict(np.load(path))
    return res, dict(CASES[name].get("env", {}), **env_extra)


def compare(dev, name):
    """Every check of one case: (worst err / (C u mag) per quantity, list of failures).  Does not raise."""
    ref = reference(name)
    worst = {"pose": 0.0, "rcov": 0.0, "y": 0.0, "P": 0.0}
    fails = []

    def ratio(kind, what, x, v, m_, C):
        x = np.asarray(x, np.float64)
        if x.shape != np.shape(v):
            fails.append("%s: shape %s vs reference %s" % (what, x.shape, np.shape(v)))
            return
        w = hp.worst_ratio(x, v, m_) / C
        worst[kind] = max(worst[kind], w)
        if w > 1.0:
            fails.append("%s: worst |x - ref| / (C u mag) = %.3g" % (what, w))

    for s, r in enumerate(ref["scans"]):
        if not np.array_equal(dev["%d/j" % s], r["j"]):
            fails.append("scan %d: associations %s vs reference %s" % (s, dev["%d/j" % s], r["j"]))
        if "%d/pose" % s in dev:
            if int(dev["%d/L" % s]) != r["L"]:
                fails.append("scan %d: %d lines vs reference %d" % (s, int(dev["%d/L" % s]), r["L"]))
            ratio("pose", "scan %d pose" % s, dev["%d/pose" % s], *r["pose"], r["C"])
            ratio("rcov", "scan %d robot cov" % s, dev["%d/rcov" % s], *r["rcov"], r["C"])
    last = ref["scans"][-1]
    if "end/pose" in dev:
        if int(dev["end/L"]) != last["L"]:
            fails.append("end: %d lines vs reference %d" % (int(dev["end/L"]), last["L"]))
        ratio("pose", "end pose", dev["end/pose"], *last["pose"], last["C"])
        ratio("rcov", "end robot cov", dev["end/rcov"], *last["rcov"], last["C"])
    if int(dev["L"]) != ref["L"]:
        fails.append("%d lines vs reference %d" % (int(dev["L"]), ref["L"]))
    ratio("y", "y", dev["y"], *ref["y"], ref["C"])
    if "P" in dev:
        ratio("P", "P blocks", dev["P"], *ref["P"], ref["C"])
    else:
        fails.append("P blocks: the live size differs from the reference's")
    return worst, fails


def check_exercised(dev, name, env, label, max_batch=64):
    """The case ran the path it is meant to: sweep launches and folded terms of the intended grouping, and the scan
    pattern the case is built around (from the reference's associations, equal to the device's once compare passed)."""
    ref = reference(name)
    c = case_inputs(name)
    ms = [z.shape[0] for _, z, _ in c["scans"]]
    J = [r["j"] for r in ref["scans"]]
    bounds, members = intended_grouping(ms, c["cap"], env, max_batch)
    sweeps, sweep_bytes = dev["prof"]
    n = 3.0 + 2.0 * int(dev["L"])
    terms = (sweep_bytes - sweeps * 8.0 * n * (n + 1.0)) / (32.0 * n)
    assert int(sweeps) == len(bounds) and round(terms) == sum(bounds), \
        "%s: %d sweep launches folding %.1f terms, the intended grouping has %d folding %d (%s; if the host's slot-ring or " \
        "budget sizing changed, see knobs())" % (
            label, sweeps, terms, len(bounds), sum(bounds), bounds)
    assert min(3 + 2 * r["L_before"] for r in ref["scans"] if not r["reset"]) >= OVERLAP_MIN_N or name == "reset"
    shared = max(len(g) for g in members)
    # a landmark appended by one scan of a group and matched by a later scan of the same group
    within = 0
    for g in members:
        for s in g[1:]:
            lo, hi = ref["scans"][g[0]]["L_before"], ref["scans"][s]["L_before"]
            within += int(((J[s] >= lo) & (J[s] < hi)).sum()) if hi > lo else 0
    note = "%d sweeps, %d terms, up to %d scans per sweep, %d lines matched a landmark appended earlier in their group" % (
        len(bounds), sum(bounds), shared, within)
    budget = knobs(env, max_batch)["budget"]
    if budget:
        assert shared >= 2 and within >= 1, "%s: %s" % (label, note)
    if name == "groups_nl1":
        crossed = [g for g in members if len(g) > 1 and
                   (2 + 2 * ref["scans"][g[0]]["L_before"]) // 64 != (2 + 2 * ref["scans"][g[0]]["L"]) // 64]
        assert not budget or crossed, "%s: no group's first scan crossed a 64-row tile boundary" % label
    if name in ("groups_nl1", "groups_nl63"):
        assert (3 + 2 * ref["L"]) % 64 == (1 if name == "groups_nl1" else 63)
    if name == "ragged" and knobs(env)["line_sms"] < 1:
        classes = {line_sms(m, c["cap"], knobs(env)) for m in ms if m}
        assert classes == {20, 21}, classes
        assert 0 in ms and max(ms) > 32 and 1 in ms
    if name == "reset":
        rs = [s for s, r in enumerate(ref["scans"]) if r["reset"]]
        assert rs, "%s: no reset" % label
        s = rs[0]
        g = next(g for g in members if s in g)
        assert (J[s] >= 0).sum() >= 1, "%s: the reset scan formed no terms" % label
        if budget:
            assert g.index(s) < len(g) - 1, "%s: no scan continues the group of the reset (%s)" % (label, g)
        assert sum(int((J[t] >= 0).sum()) for t in range(s + 2, len(J))) >= 8, "%s: the rebuilt map is not re-observed" % label
        note += ", reset in scan %d of group %s" % (s, g)
    if name == "deep":
        deepest = deepest_correction(members, J)
        assert deepest == 127, "%s: the deepest line corrected against %d pending terms" % (label, deepest)
        assert any(sum(int((J[s] >= 0).sum()) for s in g) % 2 for g in members), "%s: no odd group" % label
        note += ", deepest line corrected against %d pending terms" % deepest
    if name == "stale":
        assert int(dev["warm_matched"]) >= 2 * 16, "%s: warm-up matched %d lines" % (label, int(dev["warm_matched"]))
    return note


# knob -> (environment, cases): each checked against the reference on a few cases, not as a cross product
VARIANTS = {
    "default": ({}, ["groups_nl1", "groups_nl63", "ragged", "reset", "stale"]),
    "group0": ({"EKF_SWEEP_GROUP": "0"}, ["groups_nl1", "reset"]),
    "group64": ({"EKF_SWEEP_GROUP": "64"}, ["deep", "groups_nl63"]),
    "maxc8": ({"EKF_SWEEP_MAXC": "8"}, ["groups_nl1", "ragged"]),
    "shape10": ({"EKF_SWEEP_SHAPE": "10"}, ["groups_nl63"]),
    "shape11": ({"EKF_SWEEP_SHAPE": "11"}, ["groups_nl1"]),
    "line_loop1": ({"EKF_LINE_LOOP": "1"}, ["groups_nl63", "stale"]),
    "line_sms4": ({"EKF_LINE_SMS": "4"}, ["groups_nl1"]),          # memory-resident k_scan_lines2: 4 x 512 < L
    "fuse0": ({"EKF_FUSE_PREDICT": "0"}, ["groups_nl63", "reset"]),   # the carry goes through k_predict
    "exact_build": ({"EKF_LIB": "exact"}, ["groups_nl1", "stale"]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_pipeline_componentwise(libekf, variant, tmp_path):
    env, names = VARIANTS[variant]
    lib = None
    if env.get("EKF_LIB") == "exact":
        from slam_ros_b200 import build as b
        lib = b.build_variant("exact")
        env = {}
    for name in names:
        dev, run_env = _spawn(name, env, tmp_path, lib)
        worst, fails = compare(dev, name)
        assert not fails, "%s / %s: %d failures, first: %s" % (variant, name, len(fails), fails[:5])
        note = check_exercised(dev, name, run_env, "%s / %s" % (variant, name))
        print("pipeline componentwise %-11s %-12s worst err/(C u mag): pose %.2e  robot cov %.2e  y %.2e  P %.2e  (C = %d; %s)"
              % (variant, name, worst["pose"], worst["rcov"], worst["y"], worst["P"], reference(name)["C"], note))


# ---- mutants: one per group invariant (DESIGN section 5) ------------------------------------------------------------
# (file, anchor, replacement, invariant, case meant to catch it).  Each changes values only: no index, size, loop bound,
# barrier, event wait or stream order, so none can fault, hang or race.  The wait behind invariant 3 (grp_may_reset) is
# deliberately not mutated: without it the result is a race, not a deterministic wrong value.
MUTANTS = {
    "M1": ("ekf_api.cu", "keep ? ctx->Pbuf[ctx->rd] : 0", "0",
           "1: the new columns are seen by the group's next scan", "groups_nl1"),
    "M2": ("ekf_kernels.cu", "const int pcnt = prev_cnt_ptr ? *prev_cnt_ptr : 0;", "const int pcnt = 0;",
           "2: a term is zero at the rows appended after it", "stale"),
    "M3": ("ekf_kernels.cu", "view->cnt = reset ? 0 : b.pidx[m] - st->pbase;", "view->cnt = b.pidx[m] - st->pbase;",
           "3: a reset inside a group", "reset"),          # unobservable: see UNOBSERVABLE
    "M4": ("ekf_api.cu", "const int* carry = joins ? &ctx->d_view[par].cnt : 0;", "const int* carry = 0;",
           "a group's sweep folds every scan's terms", "groups_nl1"),
    "M5": ("ekf_api.cu", "ctx->pg_valid ? &ctx->d_view[par ^ 1].cnt : 0, ctx->peers_ok", "0, ctx->peers_ok",
           "the line loop corrects against the terms of the sweep in flight", "groups_nl1"),
}


# Mutants whose removal leaves every value unchanged.  M3: the old map's terms that a continuing scan then carries are
# zeroed by k_end_scan_a at every row the rebuilt map appends while the group is open (the group's own slots, invariant
# 2), and rows 0-2 and the 2x2 diagonal blocks are hot storage that pending terms never touch; so they contribute exactly
# zero wherever anything reads.  Measured: the reset case gives the same worst ratios with and without the mutant.
# Kept as a strict xfail: a change that makes the invariant observable turns it into a failure here.
UNOBSERVABLE = {"M3": "the carried terms of the old map are zero at every live non-hot entry (DESIGN section 5)"}


def test_mutant_anchors_occur_exactly_once():
    """A refactor that moves or rewrites one of the guarded lines breaks the mutant list here, not silently."""
    for key, (fname, anchor, repl, what, case) in MUTANTS.items():
        with open(os.path.join(CSRC, fname)) as fh:
            n = fh.read().count(anchor)
        assert n == 1, "%s: anchor %r occurs %d times in %s" % (key, anchor, n, fname)
        assert case in CASES


def build_mutant(key, workdir, table=None, count=1):
    """Copies slam_ros_b200/csrc and include (same relative layout), applies mutant `key` of `table` (default MUTANTS:
    (file, anchor, replacement, ...)) at the `count` occurrences of its anchor, starts nvcc.  Returns (process, library
    path)."""
    from slam_ros_b200 import build as b
    fname, anchor, repl = (table or MUTANTS)[key][:3]
    src = os.path.join(workdir, "slam_ros_b200", "csrc")
    shutil.copytree(CSRC, src)
    shutil.copytree(os.path.join(ROOT, "include"), os.path.join(workdir, "include"))
    path = os.path.join(src, fname)
    with open(path) as fh:
        text = fh.read()
    assert text.count(anchor) == count, (key, anchor, text.count(anchor))
    with open(path, "w") as fh:
        fh.write(text.replace(anchor, repl))
    out = os.path.join(workdir, "libekfcuda_%s.so" % key)
    cmd = [b.nvcc_path()] + b.NVCC_FLAGS + [os.path.join(src, s) for s in b.SOURCES] + ["-o", out, "-ldl"]
    return subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True), out


@pytest.fixture(scope="module")
def mutant_libs(tmp_path_factory):
    """All mutants, compiled side by side."""
    procs = {k: build_mutant(k, str(tmp_path_factory.mktemp("mutant_" + k))) for k in MUTANTS}
    libs = {}
    for k, (p, out) in procs.items():
        log, _ = p.communicate(timeout=1800)
        assert p.returncode == 0, "%s: nvcc failed\n%s" % (k, log[-3000:])
        libs[k] = out
    return libs


@pytest.mark.gpu
@pytest.mark.parametrize("key", [pytest.param(k, marks=pytest.mark.xfail(strict=True, reason=UNOBSERVABLE[k]))
                                 if k in UNOBSERVABLE else k for k in MUTANTS])
def test_each_pipeline_invariant_is_guarded(libekf, mutant_libs, key, tmp_path):
    fname, anchor, repl, what, case = MUTANTS[key]
    dev, _ = _spawn(case, {}, tmp_path, mutant_libs[key])
    worst, fails = compare(dev, case)
    print("mutant %s (invariant %s) on case %s: %d failures; worst err/(C u mag): pose %.2e  robot cov %.2e  y %.2e  P %.2e; "
          "first: %s" % (key, what, case, len(fails), worst["pose"], worst["rcov"], worst["y"], worst["P"],
                         fails[0] if fails else "-"))
    assert fails, "mutant %s (%s -> %s) passes case %s: invariant %s is not guarded" % (key, anchor, repl, case, what)
