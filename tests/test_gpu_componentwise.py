"""libekfcuda against the extended-precision reference (tests/hp_reference.py), element by element.

Every covariance entry is checked against its own magnitude, |x - ref| <= C u mag(x), not against max|P|: most of
this filter's covariance (the landmark-angle rows) is many decades below max|P|, where a normwise 1e-9 check cannot
see a missing or misplaced rank-2 term.  Associations and the number of landmarks must be identical.  Each run starts
from an uploaded state (same doubles on both sides) whose P spans 8 decades, at map sizes that put the sweep's edge
tiles at their extremes: nl = 3 + 2L = 1 and 63 (mod 64), n = 3 + 2 cap = 255 (mod 256) with cap = L, the
register-resident bound of the cluster line loop (4096 landmarks) and the overlapped two-stream path (n >= 6000).
The library runs in subprocesses so that every environment knob and the `exact` build are checked against the same
reference run.
"""
import functools
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import hp_reference as hp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TESTS = os.path.dirname(os.path.abspath(__file__))
FULL_MAX = 1100             # compare every element up to this live size; sampled tiles above
M_LIST = [1, 2, 7, 8, 9, 13, 16, 17, 31, 32, 33, 40, 64]
U_STEP = (0.02, 0.0, 0.01)


# ---- the cases: (L, cap, headroom, scans as (m matched, unmatched)) ------------------------------------------------
CASES = {
    "nl1_small": (95, 140, 0, [(m, 0) for m in M_LIST] + [(9, 3)]),
    "nl63_small": (94, 140, 0, [(m, 0) for m in M_LIST] + [(9, 3)]),
    "nl1_large": (1503, 1530, 0, [(8, 0), (40, 0), (13, 2)]),
    "nl63_large": (1502, 1530, 0, [(8, 0), (40, 0), (13, 2)]),
    "pad255": (126, 126, 0, [(7, 0), (17, 0), (33, 0), (64, 0)]),
    "pad511": (254, 254, 0, [(9, 0), (32, 0), (40, 0)]),
    "loop4096": (4096, 4100, 0, [(8, 0), (40, 0)]),
    "loop4097": (4097, 4100, 0, [(8, 0), (33, 0)]),
    "overlap2999": (2999, 3010, 0, [(8, 0), (40, 0), (12, 4)]),
    "overlap3007": (3007, 3020, 0, [(8, 0), (40, 0), (12, 4)]),
    "empty": (0, 64, 0, [(0, 20), (8, 3), (17, 2), (9, 0)]),
}


def case_inputs(name):
    """Start state and the scans' inputs, deterministic in the case name."""
    L, cap, headroom, scans = CASES[name]
    seed = sum(map(ord, name))
    rng = np.random.default_rng(seed)
    y, P, world = hp.spread_state(L, cap, seed)
    if L == 0:
        world = hp.spread_state(40, 40, seed)[2]
        y = np.zeros(3 + 2 * cap); P = np.zeros((3 + 2 * cap,) * 2); P[0, 0] = P[1, 1] = 0.05
    pose = tuple(y[:3])
    inputs = []
    known = L
    for m, extra in scans:
        pose = hp.predicted_pose(pose, U_STEP)
        if L == 0:
            ids = list(rng.permutation(known)[:m]) if known else []
            new = list(range(known, known + extra))
            z, R = hp.lines_for(world, pose, ids + new, rng)
            known += extra
        else:
            ids = rng.choice(L, m, replace=False)
            z, R = hp.lines_for(world, pose, ids, rng, n_unmatched=extra)
        inputs.append((np.array(U_STEP), z, R))
    return dict(L=L, cap=cap, headroom=headroom, y=y, P=P, scans=inputs)


def blocks_for(nl, seed=0):
    """(r0, c0, nr, nc) blocks compared at live size nl."""
    if nl <= FULL_MAX:
        return [(0, 0, nl, nl)]
    t = 64 * ((nl - 1) // 64)
    out = [(0, 0, 3, nl), (t, 0, nl - t, nl), (0, t, nl, nl - t)]
    out += [(d, d, min(64, nl - d), min(64, nl - d)) for d in range(0, nl, 64)]
    rng = np.random.default_rng(seed)
    for _ in range(32):
        r0, c0 = (int(v) * 64 for v in rng.integers(0, (nl - 1) // 64 + 1, 2))
        out.append((r0, c0, min(64, nl - r0), min(64, nl - c0)))
    return out


# ---- device side (runs in a subprocess) ---------------------------------------------------------------------------
def device_run(names, out_path, flags=0):
    from slam_ros_b200 import EkfFilter
    res = {}
    for name in names:
        c = case_inputs(name)
        f = EkfFilter(capacity_lines=c["cap"], reset_headroom=c["headroom"], flags=flags)
        f.upload(c["y"], c["P"], c["L"])
        for s, (u, z, R) in enumerate(c["scans"]):
            rc, j, pose = f.scan(u, z, R)
            res["%s/%d/j" % (name, s)] = j
            res["%s/%d/pose" % (name, s)] = pose
            res["%s/%d/y" % (name, s)] = f.download_y()
            if s == len(c["scans"]) - 1 or name.startswith("overlap"):
                nl = 3 + 2 * f.lines
                res["%s/%d/P" % (name, s)] = np.concatenate(
                    [f.download_block(*b).ravel() for b in blocks_for(nl, s)])
        f.close()
    np.savez(out_path, **res)


def device_every_count(out_path):
    """Every pending count 1..64 through the stand-alone-sized map: fresh upload, one scan of m matched lines."""
    from slam_ros_b200 import EkfFilter
    c = case_inputs("nl63_small")
    res = {}
    f = EkfFilter(capacity_lines=c["cap"], reset_headroom=0)
    for m in range(1, 65):
        z, R = _every_count_lines(m)
        f.upload(c["y"], c["P"], c["L"])
        rc, j, pose = f.scan(np.array(U_STEP), z, R)
        y, P, L = f.download_live()
        res["%d/j" % m] = j; res["%d/y" % m] = y; res["%d/P" % m] = P; res["%d/pose" % m] = pose
    f.close()
    np.savez(out_path, **res)


def _every_count_lines(m):
    L, cap, headroom, scans = CASES["nl63_small"]
    c_seed = sum(map(ord, "nl63_small"))
    world = hp.spread_state(L, cap, c_seed)[2]
    rng = np.random.default_rng(1000 + m)
    pose = hp.predicted_pose((0.3, -0.2, 0.1), U_STEP)
    return hp.lines_for(world, pose, rng.choice(L, m, replace=False), rng)


def _spawn(call, env_extra):
    path = "/tmp/ekf_componentwise_%d_%s.npz" % (os.getpid(), abs(hash((call, json.dumps(env_extra, sort_keys=True)))))
    code = "import sys; sys.path[:0] = [%r, %r]\nimport test_gpu_componentwise as t\n%s\n" % (ROOT, TESTS, call % path)
    env = dict(os.environ, **env_extra)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=1200, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    res = dict(np.load(path))
    os.remove(path)
    return res


# ---- reference side ---------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def reference(name):
    c = case_inputs(name)
    f = hp.HPFilter(c["cap"], reset_headroom=c["headroom"])
    if c["L"]:
        f.upload(c["y"], c["P"], c["L"])
    out = {}
    for s, (u, z, R) in enumerate(c["scans"]):
        st, j = f.scan(u, z, R)
        out["%s/%d/j" % (name, s)] = j
        out["%s/%d/pose" % (name, s)] = (f.pose.copy(), f.mpose.copy(), f.C)
        out["%s/%d/y" % (name, s)] = (f.y[:f.nl].copy(), f.my[:f.nl].copy(), f.C)
        if s == len(c["scans"]) - 1 or name.startswith("overlap"):
            vals, mags = [], []
            for (r0, c0, nr, nc) in blocks_for(f.nl, s):
                v, m_ = f.block(np.arange(r0, r0 + nr), np.arange(c0, c0 + nc))
                vals.append(v.ravel()); mags.append(m_.ravel())
            out["%s/%d/P" % (name, s)] = (np.concatenate(vals), np.concatenate(mags), f.C)
    assert f.min_margin >= 1e-6, "%s: a gate decision within 1e-6 of the threshold (%g)" % (name, f.min_margin)
    return out


@functools.lru_cache(maxsize=None)
def reference_every_count(m):
    c = case_inputs("nl63_small")
    f = hp.HPFilter(c["cap"], reset_headroom=0)
    f.upload(c["y"], c["P"], c["L"])
    z, R = _every_count_lines(m)
    st, j = f.scan(np.array(U_STEP), z, R)
    y, my, Pv, Pm = f.live()
    assert f.min_margin >= 1e-6
    return j, (f.pose, f.mpose), (y, my), (Pv, Pm), f.C


def compare(dev, names, label):
    worst = {"y": 0.0, "P": 0.0, "pose": 0.0}
    matched = 0
    for name in names:
        ref = reference(name)
        for key, r in ref.items():
            kind = key.rsplit("/", 1)[1]
            d = dev[key]
            if kind == "j":
                assert np.array_equal(d, r), "%s %s: associations %s vs reference %s" % (label, key, d, r)
                matched += int((r >= 0).sum())
                continue
            v, m_, C = r
            assert d.shape == v.shape, "%s %s: shape" % (label, key)
            worst[kind] = max(worst[kind], hp.check(d, v, m_, C, "%s %s" % (label, key)) / C)
    print("componentwise %-24s worst err/(C u mag): y %.2e  pose %.2e  P %.2e  (%d matched lines)"
          % (label, worst["y"], worst["pose"], worst["P"], matched))
    return matched


DEFAULT_CASES = list(CASES)
# knob -> (environment, flags, cases): each checked against the reference at a few sizes, not as a cross-product
VARIANTS = {
    "default": ({}, 0, DEFAULT_CASES),
    "shape9": ({"EKF_SWEEP_SHAPE": "9"}, 0, ["nl1_small", "nl63_large", "pad511"]),
    "shape10": ({"EKF_SWEEP_SHAPE": "10"}, 0, ["nl1_small", "nl63_large", "pad511"]),
    "shape11": ({"EKF_SWEEP_SHAPE": "11"}, 0, ["nl1_small", "nl63_large", "pad511"]),
    "dmma_nosplit": ({"EKF_DMMA_SPLIT": "0"}, 0, ["nl63_small", "nl1_large"]),
    "line_loop1": ({"EKF_LINE_LOOP": "1"}, 0, ["nl63_small", "loop4097", "overlap3007"]),
    "eager": ({}, 1, ["nl1_small", "overlap2999"]),
    "sweep_direct": ({}, 2, ["nl1_small", "nl63_large"]),
    "per_line": ({}, 4, ["nl63_small", "overlap2999"]),
    "no_overlap": ({}, 8, ["overlap2999", "overlap3007"]),
    "exact_build": ({"EKF_LIB": "exact"}, 0, ["nl1_small", "nl63_large", "overlap3007", "empty"]),
}


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_single_filter_componentwise(libekf, variant):
    env, flags, names = VARIANTS[variant]
    if env.get("EKF_LIB") == "exact":
        from slam_ros_b200 import build as b
        env = dict(env, EKF_LIB=b.build_variant("exact"))
    dev = _spawn("t.device_run(%r, %%r, flags=%d)" % (names, flags), env)
    matched = compare(dev, names, variant)
    assert matched > 20


@pytest.mark.parametrize("maxc", [8, 16, 32])
def test_sweep_every_pending_count_with_real_terms(libekf, maxc):
    """The real-term counterpart of the zero-term ring test: every pending count 1..64 at every pass width, on a map
    whose last tile is one row short of full (nl = 191)."""
    dev = _spawn("t.device_every_count(%r)", {"EKF_SWEEP_MAXC": str(maxc)})
    worst = 0.0
    for m in range(1, 65):
        j, (pv, pm), (yv, ym), (Pv, Pm), C = reference_every_count(m)
        assert np.array_equal(dev["%d/j" % m], j), (m, dev["%d/j" % m], j)
        assert (j >= 0).sum() >= m - 1
        hp.check(dev["%d/pose" % m], pv, pm, C, "m=%d pose" % m)
        hp.check(dev["%d/y" % m], yv, ym, C, "m=%d y" % m)
        worst = max(worst, hp.check(dev["%d/P" % m], Pv, Pm, C, "m=%d P" % m) / C)
    print("componentwise sweep maxc=%d, m = 1..64: worst P err/(C u mag) %.2e" % (maxc, worst))


# ---- batch filters -------------------------------------------------------------------------------------------------
B_FILTERS, B_CAP, B_WORLD = 96, 80, 75


def batch_inputs():
    """Filters seeded from the empty map and steered to map sizes 1..70 (all in one batch, one m per scan), then scans
    of m = 0, 1, 2, 3, 8, 9 lines: odd numbers of matches, and a last line that matches nothing after matches."""
    rng = np.random.default_rng(77)
    worlds = [hp.spread_state(B_WORLD, B_WORLD, 500 + f)[2] for f in range(B_FILTERS)]
    target = [1 + (f * 37) % 70 for f in range(B_FILTERS)]
    known = [0] * B_FILTERS
    poses = [(0.0, 0.0, 0.0)] * B_FILTERS
    scans = []

    def one_scan(m, plan):
        z = np.zeros((B_FILTERS, m, 2)); R = np.zeros((B_FILTERS, m, 4))
        for f in range(B_FILTERS):
            poses[f] = hp.predicted_pose(poses[f], U_STEP)
            ids = plan(f)
            if m:
                z[f], R[f] = hp.lines_for(worlds[f], poses[f], ids, rng)
        scans.append((np.tile(np.array(U_STEP), (B_FILTERS, 1)), z, R))

    def plan_for(m):
        def plan(f):
            new = min(m, max(target[f] - known[f], 0))
            if m >= 2 and new == 0 and len(scans) > 40:     # the scans after the growth end on a new landmark
                new = 1
            old = m - new
            if old > known[f]:
                old = known[f]; new = m - old
            ids = list(rng.permutation(known[f])[:old]) + list(range(known[f], known[f] + new))
            known[f] += new
            return ids
        return plan

    for _ in range(40):
        one_scan(2, plan_for(2))
    for m in (0, 1, 2, 3, 8, 9):
        one_scan(m, plan_for(m))
    return scans


def batch_device(out_path, flags=0):
    from slam_ros_b200 import EkfBatch
    bt = EkfBatch(B_FILTERS, capacity_lines=B_CAP, reset_headroom=0, flags=flags)
    res = {}
    for s, (u, z, R) in enumerate(batch_inputs()):
        rc, j, pose = bt.scan(u, z, R)
        res["%d/j" % s] = j; res["%d/pose" % s] = pose
    for f in range(B_FILTERS):
        y, P, L, pose = bt.download(f)
        res["f%d/y" % f] = y; res["f%d/P" % f] = P; res["f%d/L" % f] = np.array(L)
    bt.close()
    np.savez(out_path, **res)


@functools.lru_cache(maxsize=None)
def batch_reference():
    filters = [hp.HPFilter(B_CAP, reset_headroom=0) for _ in range(B_FILTERS)]
    J, poses = [], []
    for (u, z, R) in batch_inputs():
        J.append(np.stack([f.scan(u[i], z[i], R[i])[1] for i, f in enumerate(filters)]))
        poses.append([(f.pose.copy(), f.mpose.copy()) for f in filters])
    states = [(f.L, f.live(), f.C) for f in filters]
    assert min(f.min_margin for f in filters) >= 1e-6
    return J, poses, states


@pytest.mark.parametrize("variant", ["default", "ns3", "ns36", "ns37", "ns64", "full_gates"])
def test_batch_filters_componentwise(libekf, variant):
    env = {"EKF_BATCH_NS": variant[2:]} if variant.startswith("ns") else {}
    flags = 16 if variant == "full_gates" else 0
    dev = _spawn("t.batch_device(%%r, flags=%d)" % flags, env)
    J, poses, states = batch_reference()
    worst = 0.0
    for s in range(len(J)):
        assert np.array_equal(dev["%d/j" % s], J[s]), "scan %d" % s
        for f in range(B_FILTERS):
            pv, pm = poses[s][f]
            hp.check(dev["%d/pose" % s][f], pv, pm, states[f][2], "scan %d filter %d pose" % (s, f))
    sizes = set()
    for f in range(B_FILTERS):
        L, (yv, ym, Pv, Pm), C = states[f]
        assert int(dev["f%d/L" % f]) == L
        nl = 3 + 2 * L
        sizes.add(L)
        hp.check(dev["f%d/y" % f][:nl], yv, ym, C, "filter %d y" % f)
        worst = max(worst, hp.check(dev["f%d/P" % f][:nl, :nl], Pv, Pm, C, "filter %d P" % f) / C)
        assert not dev["f%d/P" % f][nl:].any() and not dev["f%d/P" % f][:, nl:].any()
    assert len({(3 + 2 * L) % 32 for L in sizes}) == 16, sorted(sizes)
    print("componentwise batch %-10s worst P err/(C u mag) %.2e over map sizes %d..%d" % (variant, worst, min(sizes), max(sizes)))


def test_batch_binding_accepts_empty_scans_and_early_collect(libekf):
    from slam_ros_b200 import EkfBatch
    from slam_ros_b200.ekf import EkfError, EKF_ESTATE
    bt = EkfBatch(4, capacity_lines=8)
    with pytest.raises(EkfError) as e:
        bt.collect()
    assert e.value.code == EKF_ESTATE
    rc, j, pose = bt.scan(np.tile(np.array(U_STEP), (4, 1)), np.zeros((4, 0, 2)), np.zeros((4, 0, 4)))
    assert rc == 0 and j.shape == (4, 0) and np.allclose(pose[:, 0], 0.02 * np.cos(0.005), rtol=1e-15)
    bt.submit(np.tile(np.array(U_STEP), (4, 1)), np.zeros((4, 0, 2)), np.zeros((4, 0, 4)))
    rc, j, pose = bt.collect()
    assert rc == 0 and j.shape == (4, 0)
    bt.close()


# ---- the gate at its threshold -------------------------------------------------------------------------------------
def _threshold_state(L, cap):
    """Landmark 0 at alfa = 0 with the pose at theta = 0 (cos and sin exact), the others elsewhere."""
    y, P, world = hp.spread_state(L, cap, 4242, pose=(0.0, 0.0, 0.0))
    y[3] = 0.0; y[4] = 3.0
    return y, P


def gate_device(out_path, L, cap, gates, path_name):
    from slam_ros_b200 import EkfFilter, EkfBatch
    y, P = _threshold_state(L, cap)
    z = np.array([[0.0007, 3.004]]); R = np.array([[4e-6, 0, 0, 2.5e-5]])
    res = {}
    for i, g in enumerate(map(float.fromhex, gates)):
        if path_name.startswith("batch"):
            # the batch is seeded from the empty map: one scan appends the landmark at alfa = 0
            bt = EkfBatch(2, capacity_lines=cap, gate=g, reset_headroom=0, flags=16 if path_name == "batch_full" else 0)
            bt.scan(np.zeros((2, 3)), np.tile([[[0.0, 3.0]]], (2, 1, 1)), np.tile(R, (2, 1, 1)))
            rc, j, pose = bt.scan(np.zeros((2, 3)), np.tile(z, (2, 1, 1)), np.tile(R, (2, 1, 1)))
            res[str(i)] = j[:, 0]
            bt.close()
            continue
        flags = 4 if path_name == "per_line" else 0
        f = EkfFilter(capacity_lines=cap, gate=g, reset_headroom=0, flags=flags)
        f.upload(y, P, L)
        if path_name == "associate":
            f.predict(np.zeros(3))
            j, _ = f.associate(z[0], R[0])
        else:
            rc, jj, pose = f.scan(np.zeros(3), z, R)
            j = jj[0]
        res[str(i)] = np.array([j])
        f.close()
    np.savez(out_path, **res)


@pytest.mark.parametrize("path_name", ["associate", "fused", "per_line", "overlap", "batch", "batch_full"])
def test_gate_decision_at_the_exact_threshold(libekf, path_name):
    """d^2 of the pair, computed as the reference computes it, is D; gate = sqrt(D) must accept (sqrt(D) > gate is
    false), gate = the double below must reject.  gate = inf and NaN accept every pair: the line matches landmark 0."""
    import math
    from oracle.oracle import StructuredOracle
    L, cap = (2999, 3000) if path_name == "overlap" else (5, 8)
    z = np.array([0.0007, 3.004]); R = np.array([4e-6, 0, 0, 2.5e-5])
    if path_name.startswith("batch"):
        so = StructuredOracle(cap, reset_headroom=0)
        so.scan(np.zeros(3), np.array([[0.0, 3.0]]), R[None])
        so.predict(np.zeros(3))
        D = so.gate_pair(0, z, R)[3]
    else:
        y, P = _threshold_state(L, cap)
        so = StructuredOracle(cap)
        np.ctypeslib.as_array(so._lib.ekfo_y_ptr(so._h), shape=(so.n,))[:] = y
        so.P_view()[:] = P
        import ctypes
        so._lib.ekfo_set_lines(so._h, ctypes.c_int(L))
        so.set_pose(y[:3])
        so.predict(np.zeros(3))
        D = so.gate_pair(0, z, R)[3]
    assert 0.0 < D < 1.0
    g_hi = math.sqrt(D)
    g_lo = float(np.nextafter(g_hi, 0.0))
    gates = [g_hi, g_lo, math.inf, math.nan]
    want = [0 if not (math.sqrt(abs(D)) > g) else -1 for g in gates]
    assert want[:2] == [0, -1]
    dev = _spawn("t.gate_device(%%r, %d, %d, %r, %r)" % (L, cap, [g.hex() for g in gates], path_name), {})
    for i, g in enumerate(gates):
        assert np.all(dev[str(i)] == want[i]), "%s gate=%r: %s, expected %d" % (path_name, g, dev[str(i)], want[i])
