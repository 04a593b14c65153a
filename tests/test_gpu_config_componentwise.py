"""Every max_batch regime and the other ekf_config fields against the extended-precision reference, element by element.

The other componentwise tests build their filters with the default ekf_config.  Its fields select code paths
(include/ekf.h, DESIGN sections 3-5):
  max_batch 1-15    no overlapped pipeline; the fused line loop is split every max_batch lines, each part followed by
                    an in-place sweep;
  max_batch 16-63   overlap with a smaller slot ring: group = max_batch / 2 (at most 32), ring halves at slot `group`
                    (8, 9, 17, 31: the sweep's TMA band loads start at an unaligned slot row), scans of group < m <= 32
                    lines drain and run in place;
  max_batch 65-128  no fused line loop: in-place scans go line by line (k_associate / k_gain / k_apply) and k_gain
                    corrects its column reads against up to max_batch - 1 pending terms; overlapped scans as at 64;
  max_batch > 128   the same, with more pending terms than the line loops hold (FL_MAXP).
capacity_lines 1-3, reset_headroom >= capacity_lines and encoder_noise 0 and 0.5 run from the empty map on the fused,
per-line and step-wise paths and on the batch.  First fit among several passing landmarks is set up on purpose with
duplicated landmarks, in the register- and memory-resident line loops, the per-line kernels, the overlapped path and
the batch, at the default gate and at a wide one.

Every run is compared with hp.HPFilter (associations, line count and status exact; y, pose and P within C u mag), every
max_batch run also with the default-config run on the same inputs, bit for bit (DESIGN section 4), and every case
asserts that it ran its regime (sweep launches and folded terms from profile_read, ring halves, correction depth).
test_each_config_path_is_guarded rebuilds the library with one value-only mutant and requires a failure.
"""
import functools
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import hp_reference as hp
import test_gpu_pipeline_componentwise as pcw

ROOT, TESTS, CSRC = pcw.ROOT, pcw.TESTS, pcw.CSRC
U_STEP = pcw.U_STEP
FLAG_EAGER, FLAG_PER_LINE, FLAG_NO_OVERLAP, FLAG_FULL_GATES = 1, 4, 8, 16


# ---- 1a. max_batch on a small map, in place ------------------------------------------------------------------------
SMALL_L, SMALL_CAP = 158, 200          # nl = 319 = 63 (mod 64); one scan can hold all 158 landmarks (> FL_MAXP)
MB_SMALL = [1, 2, 7, 15, 65, 100, 130]


def small_ms(mb):
    """m = 1, max_batch - 1, max_batch, max_batch + 1, 2 max_batch + 3 (capped at L) matched lines."""
    out = []
    for m in (1, mb - 1, mb, mb + 1, 2 * mb + 3):
        m = min(m, SMALL_L)
        if m >= 1 and m not in out:
            out.append(m)
    return out


@functools.lru_cache(maxsize=None)
def small_inputs(mb):
    """Start state and scans: the matched scans of small_ms(mb), then one of 5 matched and 3 unmatched lines."""
    seed = 9000 + mb
    rng = np.random.default_rng(seed)
    y, P, world = hp.spread_state(SMALL_L, SMALL_CAP, seed)
    pose, scans = tuple(y[:3]), []
    for m, extra in [(m, 0) for m in small_ms(mb)] + [(5, 3)]:
        pose = hp.predicted_pose(pose, U_STEP)
        z, R = hp.lines_for(world, pose, rng.choice(SMALL_L, m, replace=False), rng, n_unmatched=extra)
        scans.append((np.array(U_STEP), z, R))
    return dict(L=SMALL_L, cap=SMALL_CAP, headroom=0, y=y, P=P, scans=scans, world=world)


# ---- 3. the other fields, from the empty map -----------------------------------------------------------------------
# name -> (capacity_lines, reset_headroom, encoder_noise, landmarks uploaded first); FIELD_PLAN: the world lines every
# scan sees.  Encoder noise 0 starts from an uploaded map: from the empty map the heading variance would stay exactly 0,
# and the entries that are then exactly 0 come out of double arithmetic as rounding residue that no componentwise bound
# of the exact value covers (the double oracle shows the same residue).
FIELD_PLAN = [[0, 1], [0, 1, 2], [1, 2, 3, 0], [], [2, 3], [0, 1, 2, 3, 4], [4, 0]]
FIELD_CASES = {
    "cap1": (1, 0, 0.024, 0),
    "cap2": (2, 0, 0.024, 0),
    "cap3": (3, 0, 0.024, 0),
    "cap3_headroom3": (3, 3, 0.024, 0),      # headroom == capacity: every scan that ends with a landmark resets
    "cap2_headroom5": (2, 5, 0.024, 0),      # headroom > capacity: L > cap - headroom holds at L = 0 as well
    "enc0": (8, 0, 0.0, 3),
    "enc05": (8, 0, 0.5, 0),
}
FIELD_FILTERS = 4                         # the batch runs this many filters, each on a world of its own


@functools.lru_cache(maxsize=None)
def field_inputs(name, f=0):
    cap, headroom, enc, L0 = FIELD_CASES[name]
    seed = sum(map(ord, name)) + 101 * f
    rng = np.random.default_rng(seed)
    y, P, world0 = hp.spread_state(L0, cap, seed)
    world = np.concatenate([world0, hp.spread_state(6 - L0, 6 - L0, seed + 1)[2]])
    pose, scans = tuple(y[:3]) if L0 else (0.0, 0.0, 0.0), []
    for ids in FIELD_PLAN:
        pose = hp.predicted_pose(pose, U_STEP)
        if ids:
            z, R = hp.lines_for(world, pose, ids, rng)
        else:
            z, R = np.zeros((0, 2)), np.zeros((0, 4))
        scans.append((np.array(U_STEP), z, R))
    return dict(cap=cap, headroom=headroom, enc=enc, scans=scans, start=(y, P, L0) if L0 else None)


# ---- 4. first fit among several passers: duplicated landmarks ------------------------------------------------------
# name -> (L, extra capacity, gate, repeats of the duplicated line, other matched lines)
DUP_CASES = {
    "dup4096": (4096, 8, 0.4, 4, 6),       # the cluster line loop's register-resident bound
    "dup4097": (4097, 8, 0.4, 4, 6),       # one more: memory-resident, thread 0 owns copies 0 and 4096
    "dup_wide": (600, 8, 2.5, 2, 6),       # a gate at which unrelated landmarks pass as well
}
DUP_STRIDE = 256                           # copies at 0, 256, 512, ...: any line-loop stride (CTAs x 256 or 512) puts two in one thread


def dup_copies(L):
    return list(range(0, L, DUP_STRIDE))


@functools.lru_cache(maxsize=None)
def dup_inputs(name):
    """Landmark 0 copied to every DUP_STRIDE-th index (its y and its rows of P, plus 1e-6 of its diagonal block so that P
    stays positive definite, and 1e-9 rad / 1e-9 m on y: far below the lines' noise).  One scan: the line of landmark 0
    `repeats` times among `others` lines of other landmarks; then a scan that sees the duplicated line once more."""
    L, extra, gate, repeats, others = DUP_CASES[name]
    cap = L + extra
    seed = sum(map(ord, name))
    rng = np.random.default_rng(seed)
    y, P, world = hp.spread_state(L, cap, seed)
    copies = dup_copies(L)
    src = np.array([3, 4])
    for k, c in enumerate(copies[1:], 1):
        a = np.array([3 + 2 * c, 4 + 2 * c])
        P[a, :] = P[src, :]
        P[:, a] = P[:, src]
        y[a] = y[src] + 1e-9 * k
        world[c] = world[0]
    for c in copies:
        a = np.array([3 + 2 * c, 4 + 2 * c])
        for d in copies:
            b = np.array([3 + 2 * d, 4 + 2 * d])
            P[np.ix_(a, b)] = P[np.ix_(src, src)]
    for c in copies[1:]:
        a = np.array([3 + 2 * c, 4 + 2 * c])
        P[a, a] *= 1.0 + 1e-6
    pool = [i for i in range(1, L) if i not in set(copies)]
    pose, scans, seen = tuple(y[:3]), [], []
    for first in (True, False):
        ids = [0] * repeats + [int(i) for i in rng.choice(pool, others, replace=False)] if first else [0, int(rng.choice(pool))]
        ids = [int(i) for i in rng.permutation(ids)]
        pose = hp.predicted_pose(pose, U_STEP)
        z, R = hp.lines_for(world, pose, ids, rng)
        scans.append((np.array(U_STEP), z, R))
        seen.append(ids)
    return dict(L=L, cap=cap, headroom=0, gate=gate, y=y, P=P, scans=scans, copies=copies, ids=seen)


def dup_blocks(name, nl):
    """Blocks compared at live size nl: the rows of every copy and of every landmark a line observes, the robot rows,
    the diagonal tiles and sampled tiles (all of P up to pcw.FULL_MAX)."""
    c = dup_inputs(name)
    rows = set(c["copies"]) | {i for ids in c["ids"] for i in ids}
    return pcw.blocks_for(nl, rows, 7)


# batch: B_DUP filters seeded from the empty map; the first scan appends B_DUP_L lines, the line of world landmark 0 at
# every index in B_DUP_AT (three rounds of 32 landmarks), the second sees that line three times
B_DUP, B_DUP_L, B_DUP_AT = 4, 70, (3, 35, 67)


@functools.lru_cache(maxsize=None)
def batch_dup_inputs():
    rng = np.random.default_rng(4711)
    scans = []
    worlds = [hp.spread_state(B_DUP_L + 1, B_DUP_L + 1, 600 + f)[2] for f in range(B_DUP)]
    pose = (0.0, 0.0, 0.0)
    plans = [[0 if i in B_DUP_AT else i + 1 for i in range(B_DUP_L)], None]
    for s, plan in enumerate(plans):
        pose = hp.predicted_pose(pose, U_STEP)
        m = B_DUP_L if s == 0 else 9
        z = np.zeros((B_DUP, m, 2)); R = np.zeros((B_DUP, m, 4))
        for f in range(B_DUP):
            ids = plan if plan else list(rng.permutation([0, 0, 0] + [int(i) + 1 for i in rng.choice(
                [i for i in range(B_DUP_L) if i not in B_DUP_AT], 6, replace=False)]))
            z[f], R[f] = hp.lines_for(worlds[f], pose, ids, rng)
            if s == 0:
                for k, i in enumerate(B_DUP_AT):          # the copies: the same line, 1e-9 apart
                    z[f, i] = z[f, B_DUP_AT[0]] + 1e-9 * k
        scans.append((np.tile(np.array(U_STEP), (B_DUP, 1)), z, R))
    return scans


# ---- reference side -----------------------------------------------------------------------------------------------
class CountingHP(hp.HPFilter):
    """hp.HPFilter that records, for every line it gates, how many unmatched landmarks pass (nonsingular, d <= gate)."""

    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.passers = []

    def _first_fit(self, z, R):
        js, d2, rec = self.gates(z, R)
        if js.size:
            with np.errstate(invalid="ignore"):
                ok = (rec["det"] != 0) & ~(np.sqrt(np.abs(d2)) > hp.LD(self.gate))
            self.passers.append(int(ok.sum()))
        else:
            self.passers.append(0)
        return super()._first_fit(z, R)


def _run_reference(f, scans, blocks=None):
    """blocks(nl): the (r0, c0, nr, nc) blocks of P to form (raveled and concatenated); default the whole live P."""
    out = []
    for u, z, R in scans:
        st, j = f.scan(u, z, R)
        out.append(dict(st=st, j=j, L=f.L, pose=(f.pose.copy(), f.mpose.copy()), C=f.C))
    assert f.min_margin >= 1e-6, "a gate decision within 1e-6 of the threshold (%g)" % f.min_margin
    if blocks is None:
        y, my, Pv, Pm = f.live()
    else:
        y, my = f.y[:f.nl].copy(), f.my[:f.nl].copy()
        vals, mags = [], []
        for r0, c0, nr, nc in blocks(f.nl):
            v, m_ = f.block(np.arange(r0, r0 + nr), np.arange(c0, c0 + nc))
            vals.append(v.ravel()); mags.append(m_.ravel())
        Pv, Pm = np.concatenate(vals), np.concatenate(mags)
    return dict(scans=out, L=f.L, y=(y, my), P=(Pv, Pm), C=f.C, passers=list(f.passers))


@functools.lru_cache(maxsize=None)
def reference_small(mb):
    c = small_inputs(mb)
    f = CountingHP(c["cap"], reset_headroom=0)
    f.upload(c["y"], c["P"], c["L"])
    return _run_reference(f, c["scans"])


@functools.lru_cache(maxsize=None)
def reference_field(name, f=0):
    c = field_inputs(name, f)
    flt = CountingHP(c["cap"], encoder_noise=c["enc"], reset_headroom=c["headroom"])
    if c["start"]:
        flt.upload(*c["start"])
    return _run_reference(flt, c["scans"])


@functools.lru_cache(maxsize=None)
def reference_dup(name):
    c = dup_inputs(name)
    f = CountingHP(c["cap"], gate=c["gate"], reset_headroom=0)
    f.upload(c["y"], c["P"], c["L"])
    ref = _run_reference(f, c["scans"], lambda nl: dup_blocks(name, nl))
    rep = [i for i, w in enumerate(c["ids"][0]) if w == 0]                     # the repeats of landmark 0
    for i in rep:
        assert ref["passers"][i] >= 2, "%s: repeat %d had %d passers" % (name, i, ref["passers"][i])
    j = ref["scans"][0]["j"]
    if c["gate"] < 1:
        # each repeat takes the next lowest unmatched copy
        assert list(j[rep]) == c["copies"][:len(rep)], (name, j[rep])
    return ref


@functools.lru_cache(maxsize=None)
def reference_batch_dup(gate):
    filters = [CountingHP(B_DUP_L + 10, gate=gate, reset_headroom=0) for _ in range(B_DUP)]
    J, poses = [], []
    for u, z, R in batch_dup_inputs():
        J.append(np.stack([f.scan(u[i], z[i], R[i])[1] for i, f in enumerate(filters)]))
        poses.append([(f.pose.copy(), f.mpose.copy()) for f in filters])
    for f in filters:
        assert f.min_margin >= 1e-6, f.min_margin
        assert f.L >= max(B_DUP_AT) + 1
    if gate < 1:
        for f in range(B_DUP):
            rows = [i for i in range(J[1].shape[1]) if J[1][f, i] in B_DUP_AT]
            assert [int(J[1][f, i]) for i in rows] == list(B_DUP_AT), (f, J[1][f])
    for flt in filters:
        reps = [p for p in flt.passers[-9:] if p >= 2]
        assert len(reps) >= 2, flt.passers[-9:]
    return J, poses, [(f.L, f.live(), f.C) for f in filters]


# ---- device side (runs in a subprocess) ----------------------------------------------------------------------------
def _filter_run(res, key, f, scans, path, prof=True):
    """Runs `scans` on filter f by `path` (scan, stepwise, device); results under key/..."""
    if prof:
        f.profile_enable(True)
    if path == "device":
        import torch
        dev = torch.device("cuda")
        js = []
        for u, z, R in scans:
            m = z.shape[0]
            d_u = torch.tensor(u, device=dev); d_z = torch.tensor(z, device=dev); d_R = torch.tensor(R, device=dev)
            d_j = torch.full((max(m, 1),), -7, dtype=torch.int32, device=dev)
            f.scan_device(d_u.data_ptr(), m, d_z.data_ptr(), d_R.data_ptr(), d_j.data_ptr())
            js.append((d_j, m, d_u, d_z, d_R))
        f.sync()
        for s, (d_j, m, *_) in enumerate(js):
            res["%s/%d/j" % (key, s)] = d_j.cpu().numpy()[:m]
        pose, L, st = f.state()
        res["%s/end/pose" % key] = pose
    else:
        for s, (u, z, R) in enumerate(scans):
            if path == "stepwise":
                f.predict(u)
                j = np.full(z.shape[0], -1, np.int32)
                for i in range(z.shape[0]):
                    j[i], _ = f.associate(z[i], R[i])
                    if j[i] >= 0:
                        f.update(int(j[i]), z[i], R[i])
                    else:
                        f.add_line(z[i], R[i])
                rc, pose = f.end_scan(z.shape[0])
            else:
                rc, j, pose = f.scan(u, z, R)
            res["%s/%d/j" % (key, s)] = j; res["%s/%d/pose" % (key, s)] = pose
            res["%s/%d/st" % (key, s)] = np.array(rc); res["%s/%d/L" % (key, s)] = np.array(f.lines)
    if prof:
        p = f.profile_read()
        f.profile_enable(False)
        res["%s/prof" % key] = np.array([p["sweeps"], p["sweep_bytes"]])
    y, P, L = f.download_live()
    res["%s/y" % key] = y; res["%s/P" % key] = P; res["%s/L" % key] = np.array(L)


def _grow_line_tables(f, n):
    """A fused scan of n lines on the empty map: the step-wise calls then accept scans of up to n lines (ekf.h)."""
    z = np.zeros((n, 2)); z[:, 0] = np.linspace(-3.0, 3.0, n); z[:, 1] = 4.0
    R = np.tile([4e-6, 0.0, 0.0, 2.5e-5], (n, 1))
    f.scan(np.zeros(3), z, R)


def small_device(out_path, path, mbs):
    from slam_ros_b200 import EkfFilter
    res = {}
    flags = {"fused": 0, "device": 0, "stepwise": 0, "per_line": FLAG_PER_LINE, "eager": FLAG_EAGER}[path]
    for mb in mbs:
        c = small_inputs(mb)
        for cfg_mb in (mb, 64):
            f = EkfFilter(capacity_lines=c["cap"], reset_headroom=0, max_batch=cfg_mb, flags=flags)
            if path == "stepwise":
                _grow_line_tables(f, SMALL_L + 8)
            f.upload(c["y"], c["P"], c["L"])
            _filter_run(res, "%d/%d" % (mb, cfg_mb), f, c["scans"], "device" if path == "device" else path)
            f.close()
    np.savez(out_path, **res)


def field_cases(path):
    """The batch starts from the empty map only (it has no upload)."""
    return [n for n in FIELD_CASES if not (path.startswith("batch") and FIELD_CASES[n][3])]


def field_device(out_path, path):
    from slam_ros_b200 import EkfFilter, EkfBatch
    res = {}
    for name in field_cases(path):
        c = field_inputs(name)
        if path.startswith("batch"):
            bt = EkfBatch(FIELD_FILTERS, capacity_lines=c["cap"], encoder_noise=c["enc"], reset_headroom=c["headroom"],
                          flags=FLAG_FULL_GATES if path == "batch_full" else 0)
            per = [field_inputs(name, f)["scans"] for f in range(FIELD_FILTERS)]
            for s in range(len(per[0])):
                u = np.stack([p[s][0] for p in per]); z = np.stack([p[s][1] for p in per]); R = np.stack([p[s][2] for p in per])
                rc, j, pose = bt.scan(u, z, R)
                res["%s/%d/j" % (name, s)] = j; res["%s/%d/pose" % (name, s)] = pose
            for f in range(FIELD_FILTERS):
                y, P, L, pose = bt.download(f)
                res["%s/f%d/y" % (name, f)] = y; res["%s/f%d/P" % (name, f)] = P; res["%s/f%d/L" % (name, f)] = np.array(L)
            bt.close()
            continue
        f = EkfFilter(capacity_lines=c["cap"], encoder_noise=c["enc"], reset_headroom=c["headroom"],
                      flags=FLAG_PER_LINE if path == "per_line" else 0)
        if c["start"]:
            f.upload(*c["start"])
        _filter_run(res, name, f, c["scans"], path, prof=False)
        f.close()
    np.savez(out_path, **res)


def dup_device(out_path, names, flags=0):
    from slam_ros_b200 import EkfFilter
    res = {}
    for name in names:
        c = dup_inputs(name)
        f = EkfFilter(capacity_lines=c["cap"], gate=c["gate"], reset_headroom=0, flags=flags)
        f.upload(c["y"], c["P"], c["L"])
        for s, (u, z, R) in enumerate(c["scans"]):
            rc, j, pose = f.scan(u, z, R)
            res["%s/%d/j" % (name, s)] = j; res["%s/%d/pose" % (name, s)] = pose
            res["%s/%d/st" % (name, s)] = np.array(rc); res["%s/%d/L" % (name, s)] = np.array(f.lines)
        res["%s/y" % name] = f.download_y()
        L = f.lines
        res["%s/L" % name] = np.array(L)
        res["%s/P" % name] = np.concatenate([f.download_block(*b).ravel() for b in dup_blocks(name, 3 + 2 * L)])
        f.close()
    np.savez(out_path, **res)


def batch_dup_device(out_path, gate, flags=0):
    from slam_ros_b200 import EkfBatch
    bt = EkfBatch(B_DUP, capacity_lines=B_DUP_L + 10, gate=gate, reset_headroom=0, flags=flags)
    res = {}
    for s, (u, z, R) in enumerate(batch_dup_inputs()):
        rc, j, pose = bt.scan(u, z, R)
        res["%d/j" % s] = j; res["%d/pose" % s] = pose
    for f in range(B_DUP):
        y, P, L, pose = bt.download(f)
        res["f%d/y" % f] = y; res["f%d/P" % f] = P; res["f%d/L" % f] = np.array(L)
    bt.close()
    np.savez(out_path, **res)


def _spawn(call, env_extra, workdir, lib=None):
    path = os.path.join(str(workdir), "cfg_%s.npz" % abs(hash((call, json.dumps(env_extra, sort_keys=True), lib))))
    code = "import sys; sys.path[:0] = [%r, %r]\nimport test_gpu_config_componentwise as t\n%s\n" % (
        ROOT, TESTS, call % path)
    env = dict(os.environ)
    for k in ("EKF_SWEEP_GROUP", "EKF_SWEEP_MAXC", "EKF_SWEEP_SHAPE", "EKF_LINE_LOOP", "EKF_LINE_SMS", "EKF_FUSE_PREDICT",
              "EKF_LIB", "EKF_CHUNK", "EKF_CHUNK_ABOVE", "EKF_LINE_THREADS"):
        env.pop(k, None)
    env.update(env_extra)
    if lib:
        env["EKF_LIB"] = lib
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=1800, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    return dict(np.load(path))


# ---- comparison ------------------------------------------------------------------------------------------------------
def compare_run(dev, key, ref, label, fails, worst, statuses=True):
    """dev[key/...] against a _run_reference result; appends to fails, raises nothing."""
    def ratio(kind, what, x, v, m_, C):
        x = np.asarray(x, np.float64)
        if x.shape != np.shape(v):
            fails.append("%s %s: shape %s vs reference %s" % (label, what, x.shape, np.shape(v)))
            return
        w = hp.worst_ratio(x, v, m_) / C
        worst[kind] = max(worst.get(kind, 0.0), w)
        if w > 1.0:
            fails.append("%s %s: worst |x - ref| / (C u mag) = %.3g" % (label, what, w))

    for s, r in enumerate(ref["scans"]):
        d = dev["%s/%d/j" % (key, s)]
        if not np.array_equal(d, r["j"]):
            fails.append("%s scan %d: associations %s vs reference %s" % (label, s, d, r["j"]))
        if "%s/%d/pose" % (key, s) in dev:
            ratio("pose", "scan %d pose" % s, dev["%s/%d/pose" % (key, s)], *r["pose"], r["C"])
            if int(dev["%s/%d/L" % (key, s)]) != r["L"]:
                fails.append("%s scan %d: %d lines vs reference %d" % (label, s, int(dev["%s/%d/L" % (key, s)]), r["L"]))
            if statuses and int(dev["%s/%d/st" % (key, s)]) != r["st"]:
                fails.append("%s scan %d: status %d vs reference %d" % (label, s, int(dev["%s/%d/st" % (key, s)]), r["st"]))
    if "%s/end/pose" % key in dev:
        last = ref["scans"][-1]
        ratio("pose", "end pose", dev["%s/end/pose" % key], *last["pose"], last["C"])
    if int(dev["%s/L" % key]) != ref["L"]:
        fails.append("%s: %d lines vs reference %d" % (label, int(dev["%s/L" % key]), ref["L"]))
        return
    ratio("y", "y", dev["%s/y" % key], *ref["y"], ref["C"])
    ratio("P", "P", dev["%s/P" % key], *ref["P"], ref["C"])


def bit_identical(dev, key_a, key_b):
    """Keys under key_a whose arrays differ from key_b's (profile counters excepted)."""
    out = []
    for k in dev:
        if k.startswith(key_a + "/") and not k.endswith("/prof"):
            kb = key_b + k[len(key_a):]
            if kb not in dev or dev[k].shape != dev[kb].shape or dev[k].tobytes() != dev[kb].tobytes():
                out.append(k[len(key_a) + 1:])
    return out


def folded(prof, L):
    """(sweep launches, terms they folded) from profile_read (bytes resolved at the final n, ekf_profile_read)."""
    sweeps, sweep_bytes = prof
    n = 3.0 + 2.0 * L
    return int(sweeps), int(round((sweep_bytes - sweeps * 8.0 * n * (n + 1.0)) / (32.0 * n)))


def intended_inplace(ms, matched, mb, path):
    """(sweeps, terms) of in-place scans on a non-empty map: the scan paths fold every max_batch lines (matched or not)
    and at the end; the eager sweep folds after every line; the step-wise calls count only ekf_update."""
    if path == "eager":
        return sum(ms), sum(ms)
    counts = matched if path == "stepwise" else ms
    return sum(len(pcw.inplace_bounds(m, mb)) for m in counts), sum(counts)


# ---- 1a. tests: max_batch on the small map ---------------------------------------------------------------------------
SMALL_PATHS = ["fused", "per_line", "eager", "stepwise", "device"]


def check_small(dev, path, mbs, label):
    fails, worst, notes = [], {}, []
    deepest = 0
    for mb in mbs:
        ref = reference_small(mb)
        for cfg_mb in (mb, 64):
            compare_run(dev, "%d/%d" % (mb, cfg_mb), ref, "%s max_batch=%d (inputs of %d)" % (label, cfg_mb, mb), fails,
                        worst, statuses=path != "device")
        diff = bit_identical(dev, "%d/%d" % (mb, mb), "%d/64" % mb)
        if diff:
            fails.append("%s max_batch=%d: not bit-identical to max_batch=64 in %s" % (label, mb, diff[:6]))
        ms = [z.shape[0] for _, z, _ in small_inputs(mb)["scans"]]
        matched = [int((r["j"] >= 0).sum()) for r in ref["scans"]]
        for cfg_mb in (mb, 64):
            want = intended_inplace(ms, matched, cfg_mb, path)
            got = folded(dev["%d/%d/prof" % (mb, cfg_mb)], ref["L"])
            if got != want:
                fails.append("%s max_batch=%d: %d sweeps folding %d terms, intended %d folding %d" % (
                    label, cfg_mb, got[0], got[1], want[0], want[1]))
        if path in ("per_line", "stepwise"):
            deepest = max(deepest, max(min(m, mb) - 1 for m in (matched if path == "stepwise" else ms)))
        notes.append("%d:%d sweeps" % (mb, folded(dev["%d/%d/prof" % (mb, mb)], ref["L"])[0]))
    return fails, worst, deepest, ", ".join(notes)


@pytest.mark.gpu
@pytest.mark.parametrize("path", SMALL_PATHS)
def test_max_batch_in_place_componentwise(libekf, path, tmp_path):
    dev = _spawn("t.small_device(%%r, %r, %r)" % (path, MB_SMALL), {}, tmp_path)
    fails, worst, deepest, note = check_small(dev, path, MB_SMALL, path)
    assert not fails, "%d failures, first: %s" % (len(fails), fails[:5])
    if path in ("per_line", "stepwise"):
        assert deepest > 64, "%s: the deepest k_gain corrected against %d pending terms" % (path, deepest)
    print("config componentwise max_batch in place %-9s worst err/(C u mag): %s  (%s; deepest k_gain correction %d)"
          % (path, "  ".join("%s %.2e" % kv for kv in sorted(worst.items())), note, deepest))


# ---- 1b. max_batch on the large map, overlapped ----------------------------------------------------------------------
RING_MS = [4, 4, 3, 5, 8, 9, 10, 0, 17, 18, 33, 6, 6, 31, 32, 70, 1, 1]
CONFIG_CASES = {
    # m = 0; m <= group (groups join); group < m <= 32 (drain, in place) for every group below 64; m > 32 (chunks);
    # 70 lines: without overlap one in-place sweep of the per-line path folds 65 and more terms
    "ring": dict(L=3000, cap=3070, headroom=0, plan=pcw._ragged(RING_MS)),
}
pcw.CASES.update(CONFIG_CASES)
# variant -> (ekf_config fields, case)
RING_VARIANTS = {
    "mb16": (dict(max_batch=16), "ring"),                       # ring halves at 0 and 8
    "mb18": (dict(max_batch=18), "ring"),                       # ... 9: unaligned
    "mb34_reset": (dict(max_batch=34), "reset"),                # ... 17; reset inside a group; ekf_scan_device
    "mb63_device": (dict(max_batch=63), "reset"),               # ... 31; ekf_scan_device
    "mb65": (dict(max_batch=65), "ring"),
    "mb65_no_overlap": (dict(max_batch=65, flags=FLAG_NO_OVERLAP), "ring"),
    "mb100": (dict(max_batch=100), "ring"),
    "mb100_no_overlap": (dict(max_batch=100, flags=FLAG_NO_OVERLAP), "ring"),
}


@functools.lru_cache(maxsize=None)
def _default_ring_run(name, workdir):
    return pcw._spawn(name, {}, workdir, cfg={}, module="test_gpu_config_componentwise")[0]


def check_ring(dev, name, cfg, label):
    """The regime the variant is meant to run: in place (no overlap: one sweep per max_batch lines), or the intended
    grouping of the reduced ring with at least one hand-off of more than 4 terms from an unaligned ring half."""
    mb = cfg["max_batch"]
    ref = pcw.reference(name)
    c = pcw.case_inputs(name)
    ms = [z.shape[0] for _, z, _ in c["scans"]]
    if cfg.get("flags", 0) & FLAG_NO_OVERLAP:
        want = intended_inplace(ms, None, mb, "fused")
        got = folded(dev["prof"], int(dev["L"]))
        assert got == want, "%s: %d sweeps folding %d terms, intended %d folding %d" % (label, got[0], got[1], *want)
        most = max(pcw.inplace_bounds(max(ms), mb))
        assert mb <= 64 or most > 64, "%s: no in-place sweep folded more than 64 terms" % label
        return "in place, %d sweeps, %d terms, largest sweep %d terms" % (got[0], got[1], most)
    note = pcw.check_exercised(dev, name, {}, label, max_batch=mb)
    k = pcw.knobs({}, mb)
    halves = []
    bounds, members = pcw.intended_grouping(ms, c["cap"], {}, mb, halves)
    drained = sum(1 for h in halves if h is None)
    band1 = [b for b, h in zip(bounds, halves) if h == 1 and b > 4]
    if k["group"] % 8:
        assert band1, "%s: no hand-off of more than 4 terms from the unaligned ring half at slot %d" % (label, k["group"])
    if name == "ring" and k["group"] < 32:
        assert drained >= 2, "%s: no scan drained to the in-place path" % label
    return note + "; group %d, %d in-place sweeps, %d band hand-offs from half 1 (slot %d)" % (
        k["group"], drained, len(band1), k["group"])


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(RING_VARIANTS))
def test_max_batch_overlapped_componentwise(libekf, variant, tmp_path_factory):
    cfg, name = RING_VARIANTS[variant]
    base = str(tmp_path_factory.getbasetemp())
    dev, _ = pcw._spawn(name, {}, base, cfg=cfg, module="test_gpu_config_componentwise")
    worst, fails = pcw.compare(dev, name)
    assert not fails, "%s / %s: %d failures, first: %s" % (variant, name, len(fails), fails[:5])
    note = check_ring(dev, name, cfg, "%s / %s" % (variant, name))
    ref_dev = _default_ring_run(name, base)
    diff = [k for k in dev if k not in ("prof", "warm_matched") and
            not (k in ref_dev and dev[k].shape == ref_dev[k].shape and dev[k].tobytes() == ref_dev[k].tobytes())]
    assert not diff, "%s: not bit-identical to the default config in %s" % (variant, diff[:8])
    print("config componentwise %-17s %-6s worst err/(C u mag): pose %.2e  robot cov %.2e  y %.2e  P %.2e  (%s)"
          % (variant, name, worst["pose"], worst["rcov"], worst["y"], worst["P"], note))


# ---- 3. tests: the other fields ------------------------------------------------------------------------------------------
def check_fields(dev, path):
    fails, worst = [], {}
    resets = caps = 0
    for name in field_cases(path):
        if path.startswith("batch"):
            for f in range(FIELD_FILTERS):
                ref = reference_field(name, f)
                for s, r in enumerate(ref["scans"]):
                    d = dev["%s/%d/j" % (name, s)][f]
                    if not np.array_equal(d, r["j"]):
                        fails.append("%s filter %d scan %d: associations %s vs reference %s" % (name, f, s, d, r["j"]))
                    w = hp.worst_ratio(dev["%s/%d/pose" % (name, s)][f], *r["pose"]) / r["C"]
                    worst["pose"] = max(worst.get("pose", 0.0), w)
                    if w > 1:
                        fails.append("%s filter %d scan %d pose: %.3g" % (name, f, s, w))
                L = int(dev["%s/f%d/L" % (name, f)])
                if L != ref["L"]:
                    fails.append("%s filter %d: %d lines vs reference %d" % (name, f, L, ref["L"]))
                    continue
                nl = 3 + 2 * L
                for kind, x, (v, m_) in (("y", dev["%s/f%d/y" % (name, f)][:nl], ref["y"]),
                                         ("P", dev["%s/f%d/P" % (name, f)][:nl, :nl], ref["P"])):
                    w = hp.worst_ratio(x, v, m_) / ref["C"]
                    worst[kind] = max(worst.get(kind, 0.0), w)
                    if w > 1:
                        fails.append("%s filter %d %s: %.3g" % (name, f, kind, w))
                if dev["%s/f%d/P" % (name, f)][nl:].any() or dev["%s/f%d/P" % (name, f)][:, nl:].any():
                    fails.append("%s filter %d: P written outside the live part" % (name, f))
        else:
            compare_run(dev, name, reference_field(name), "%s %s" % (path, name), fails, worst)
    for name in FIELD_CASES:
        ref = reference_field(name)
        caps += sum(r["st"] == 2 for r in ref["scans"])
        ms = [z.shape[0] for _, z, _ in field_inputs(name)["scans"]]
        resets += sum(1 for m, r in zip(ms, ref["scans"]) if m and r["L"] == 0)     # a scan with lines that ends empty
    return fails, worst, caps, resets


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["fused", "per_line", "stepwise", "batch", "batch_full"])
def test_config_fields_componentwise(libekf, path, tmp_path):
    dev = _spawn("t.field_device(%%r, %r)" % path, {}, tmp_path)
    fails, worst, caps, resets = check_fields(dev, path)
    assert not fails, "%s: %d failures, first: %s" % (path, len(fails), fails[:5])
    print("config componentwise fields %-10s worst err/(C u mag): %s  (%d scans at capacity, %d resets)"
          % (path, "  ".join("%s %.2e" % kv for kv in sorted(worst.items())), caps, resets))


# ---- 4. tests: first fit among several passers ----------------------------------------------------------------------
# variant -> (environment, flags, cases)
DUP_VARIANTS = {
    "in_place": ({}, FLAG_NO_OVERLAP, ["dup4096", "dup4097", "dup_wide"]),
    "line_loop1": ({"EKF_LINE_LOOP": "1"}, FLAG_NO_OVERLAP, ["dup4097"]),
    "per_line": ({}, FLAG_PER_LINE, ["dup4097", "dup_wide"]),
    "overlap": ({}, 0, ["dup4097"]),
    "overlap_line_sms4": ({"EKF_LINE_SMS": "4"}, 0, ["dup4097"]),   # memory-resident: 4 x 512 threads < L
}


def check_dup(dev, names, label):
    fails, worst = [], {}
    for name in names:
        ref = reference_dup(name)
        for s, r in enumerate(ref["scans"]):
            d = dev["%s/%d/j" % (name, s)]
            if not np.array_equal(d, r["j"]):
                fails.append("%s %s scan %d: associations %s vs reference %s" % (label, name, s, d, r["j"]))
            for kind, key in (("st", "st"), ("L", "L")):
                if int(dev["%s/%d/%s" % (name, s, key)]) != r[kind]:
                    fails.append("%s %s scan %d: %s %d vs %d" % (label, name, s, kind, int(dev["%s/%d/%s" % (name, s, key)]), r[kind]))
            w = hp.worst_ratio(dev["%s/%d/pose" % (name, s)], *r["pose"]) / r["C"]
            worst["pose"] = max(worst.get("pose", 0.0), w)
            if w > 1:
                fails.append("%s %s scan %d pose: %.3g" % (label, name, s, w))
        if int(dev["%s/L" % name]) != ref["L"]:
            fails.append("%s %s: %d lines vs reference %d" % (label, name, int(dev["%s/L" % name]), ref["L"]))
            continue
        w = hp.worst_ratio(dev["%s/y" % name], *ref["y"]) / ref["C"]
        worst["y"] = max(worst.get("y", 0.0), w)
        if w > 1:
            fails.append("%s %s y: %.3g" % (label, name, w))
        w = hp.worst_ratio(dev["%s/P" % name], *ref["P"]) / ref["C"]
        worst["P"] = max(worst.get("P", 0.0), w)
        if w > 1:
            fails.append("%s %s P: %.3g" % (label, name, w))
    return fails, worst


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(DUP_VARIANTS))
def test_first_fit_among_duplicates(libekf, variant, tmp_path):
    env, flags, names = DUP_VARIANTS[variant]
    dev = _spawn("t.dup_device(%%r, %r, flags=%d)" % (names, flags), env, tmp_path)
    fails, worst = check_dup(dev, names, variant)
    assert not fails, "%s: %d failures, first: %s" % (variant, len(fails), fails[:5])
    passers = {n: max(reference_dup(n)["passers"]) for n in names}
    print("config componentwise duplicates %-17s worst err/(C u mag): %s  (most passers per line: %s)"
          % (variant, "  ".join("%s %.2e" % kv for kv in sorted(worst.items())), passers))


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["default", "full_gates", "wide", "wide_full_gates"])
def test_batch_first_fit_among_duplicates(libekf, variant, tmp_path):
    gate = 2.5 if variant.startswith("wide") else 0.4
    flags = FLAG_FULL_GATES if variant.endswith("full_gates") else 0
    dev = _spawn("t.batch_dup_device(%%r, %r, flags=%d)" % (gate, flags), {}, tmp_path)
    J, poses, states = reference_batch_dup(gate)
    worst = 0.0
    for s in range(len(J)):
        assert np.array_equal(dev["%d/j" % s], J[s]), "scan %d: %s vs reference %s" % (s, dev["%d/j" % s], J[s])
        for f in range(B_DUP):
            hp.check(dev["%d/pose" % s][f], *poses[s][f], states[f][2], "scan %d filter %d pose" % (s, f))
    for f in range(B_DUP):
        L, (yv, ym, Pv, Pm), C = states[f]
        assert int(dev["f%d/L" % f]) == L
        nl = 3 + 2 * L
        hp.check(dev["f%d/y" % f][:nl], yv, ym, C, "filter %d y" % f)
        worst = max(worst, hp.check(dev["f%d/P" % f][:nl, :nl], Pv, Pm, C, "filter %d P" % f) / C)
    print("config componentwise batch duplicates %-15s worst P err/(C u mag) %.2e" % (variant, worst))


# ---- CPU tests: the sizing, the reference runs, the mutant anchors -------------------------------------------------
def test_knobs_follow_create_common():
    """pcw.knobs against sizings worked out by hand from create_common (ekf_api.cu)."""
    want = {16: (8, 16, 8, 8), 18: (9, 18, 9, 9), 34: (17, 34, 16, 16), 63: (31, 63, 16, 16), 64: (64, 128, 16, 16),
            100: (64, 128, 16, 16), 130: (64, 130, 16, 16), 2: (1, 2, 1, 1)}
    for mb, (group, slots, budget, chunk) in want.items():
        k = pcw.knobs({}, mb)
        assert (k["group"], k["slots"], k["budget"], k["chunk"]) == (group, slots, budget, chunk), (mb, k)
        assert k["overlap"] == (mb >= 16)
    assert pcw.knobs({"EKF_SWEEP_MAXC": "8"}, 100)["group"] == 16
    assert pcw.inplace_bounds(131, 65) == [65, 65, 1] and pcw.inplace_bounds(0, 7) == []
    halves = []
    b, m = pcw.intended_grouping([4, 4, 12, 40, 0, 5], 3070, {}, 18, halves)
    # 4 + 4 join (budget 9); 12 > group 9 drains (one in-place sweep); 40 runs as chunks of 9; 5 alone
    assert b == [8, 12, 9, 9, 9, 9, 4, 5] and halves == [0, None, 1, 0, 1, 0, 1, 0], (b, halves)
    assert m[0] == [0, 1] and m[1] == [2]


@pytest.mark.parametrize("mb", MB_SMALL)
def test_small_reference_runs(mb):
    ref = reference_small(mb)
    matched = [int((r["j"] >= 0).sum()) for r in ref["scans"]]
    ms = small_ms(mb)
    assert max(matched) >= min(max(ms), SMALL_L) - 8, (ms, matched)
    assert (3 + 2 * SMALL_L) % 64 == 63
    if mb >= 100:
        assert max(matched) > 128, matched
    assert ref["L"] > SMALL_L                     # the last scan's unmatched lines were appended


def test_ring_reference_run():
    ref = pcw.reference("ring")
    assert sum(int((r["j"] >= 0).sum()) for r in ref["scans"]) >= sum(RING_MS) * 3 // 4
    ms = [z.shape[0] for _, z, _ in pcw.case_inputs("ring")["scans"]]
    for mb in (16, 18, 34, 63, 65, 100):
        halves = []
        bounds, _ = pcw.intended_grouping(ms, 3070, {}, mb, halves)
        group = pcw.knobs({}, mb)["group"]
        assert any(b > 4 and h == 1 for b, h in zip(bounds, halves)), mb
        assert (None in halves) == (group < 32), (mb, halves)
    reset = [z.shape[0] for _, z, _ in pcw.case_inputs("reset")["scans"]]
    for mb in (34, 63):
        halves = []
        bounds, _ = pcw.intended_grouping(reset, 3326, {}, mb, halves)
        assert any(b > 4 and h == 1 for b, h in zip(bounds, halves)), mb


@pytest.mark.parametrize("name", list(FIELD_CASES))
def test_field_reference_runs(name):
    for f in range(FIELD_FILTERS):
        ref = reference_field(name, f)
        cap, headroom, enc, L0 = FIELD_CASES[name]
        assert sum(int((r["j"] >= 0).sum()) for r in ref["scans"]) >= 1 or headroom >= cap
        if headroom == 0 and cap <= 3:
            assert any(r["st"] == 2 for r in ref["scans"]), "%s: never at capacity" % name
        if headroom >= cap:
            assert all(r["L"] == 0 for r in ref["scans"]), "%s: a scan ended without a reset" % name


@pytest.mark.parametrize("name", list(DUP_CASES))
def test_dup_reference_runs(name):
    ref = reference_dup(name)
    assert sum(p >= 2 for p in ref["passers"]) >= DUP_CASES[name][3]


@pytest.mark.parametrize("gate", [0.4, 2.5])
def test_batch_dup_reference_runs(gate):
    reference_batch_dup(gate)


# ---- 6. mutants ------------------------------------------------------------------------------------------------------
# key -> (file, anchor, replacement, occurrences, what it breaks, how to run the case that catches it).  Each changes
# values only: no index, bound, barrier, event wait or stream order, so none can fault, hang or race.  Ma only ever moves
# a band read upward: inside half 1, into slots the ring does not use, or past the slot array, where TMA fills zeros;
# none of that memory is written while the sweep runs.
MUTANTS = {
    "Ma": ("ekf_kernels.cu", "slot0 + c0 + 8 * bi", "((slot0 + 7) & ~7) + c0 + 8 * bi", 4,
           "the sweep's band loads start at the ring half's own slot row", ("ring", "mb18")),
    "Mb": ("ekf_kernels.cu", "for (int i = 0; i < np; ++i)\n    p = sub_rank2(p, b.KSp",
           "for (int i = 0; i < np && i < 64; ++i)\n    p = sub_rank2(p, b.KSp", 1,
           "k_gain corrects its column reads against every pending term", ("small", "per_line")),
    "Mc": ("ekf_kernels.cu", "if (cand == EKF_NO_MATCH && h.mt != epoch) {", "if (h.mt != epoch) {", 1,
           "a line-loop thread keeps its first passer", ("dup", "overlap_line_sms4")),
}


def test_config_mutant_anchors():
    for key, (fname, anchor, repl, count, what, how) in MUTANTS.items():
        with open(os.path.join(CSRC, fname)) as fh:
            n = fh.read().count(anchor)
        assert n == count, "%s: anchor %r occurs %d times in %s, expected %d" % (key, anchor, n, fname, count)


@pytest.fixture(scope="module")
def config_mutant_libs(tmp_path_factory):
    procs = {k: pcw.build_mutant(k, str(tmp_path_factory.mktemp("cfg_mutant_" + k)), MUTANTS, MUTANTS[k][3])
             for k in MUTANTS}
    libs = {}
    for k, (p, out) in procs.items():
        log, _ = p.communicate(timeout=1800)
        assert p.returncode == 0, "%s: nvcc failed\n%s" % (k, log[-3000:])
        libs[k] = out
    return libs


@pytest.mark.gpu
@pytest.mark.parametrize("key", list(MUTANTS))
def test_each_config_path_is_guarded(libekf, config_mutant_libs, key, tmp_path):
    fname, anchor, repl, count, what, (kind, variant) = MUTANTS[key]
    lib = config_mutant_libs[key]
    if kind == "ring":
        cfg, name = RING_VARIANTS[variant]
        dev, _ = pcw._spawn(name, {}, str(tmp_path), lib, cfg=cfg, module="test_gpu_config_componentwise")
        worst, fails = pcw.compare(dev, name)
    elif kind == "small":
        mbs = [100, 130]
        dev = _spawn("t.small_device(%%r, %r, %r)" % (variant, mbs), {}, tmp_path, lib)
        fails, worst, _, _ = check_small(dev, variant, mbs, variant)
    else:
        env, flags, names = DUP_VARIANTS[variant]
        dev = _spawn("t.dup_device(%%r, %r, flags=%d)" % (names, flags), env, tmp_path, lib)
        fails, worst = check_dup(dev, names, variant)
    print("config mutant %s (%s) on %s: %d failures; first: %s" % (key, what, variant, len(fails), fails[0] if fails else "-"))
    assert fails, "mutant %s (%r -> %r) passes %s: '%s' is not guarded" % (key, anchor, repl, variant, what)
