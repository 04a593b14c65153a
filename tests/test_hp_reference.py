"""CPU tests of the extended-precision reference (tests/hp_reference.py) and of the association threshold.

The reference is pinned to the structured oracle: identical associations and the oracle's state within the
componentwise bound.  The fault test records why the componentwise check exists: faults a covariance sweep could
plausibly have are flagged by it while the suite's normwise 1e-9 measure lets at least one of them through.
"""
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

import hp_reference as hp
from slam_ros_b200 import scenario as sc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _pin(so, ref, what):
    yo, Po = so.live()
    yv, ym, Pv, Pm = ref.live()
    assert so.lines == ref.L, what
    hp.check(yo, yv, ym, ref.C, what + " y")
    hp.check(Po, Pv, Pm, ref.C, what + " P")
    hp.check(so.pose, ref.pose, ref.mpose, ref.C, what + " pose")


def test_precision_is_extended():
    hp.require_precision()
    assert np.finfo(np.longdouble).nmant >= 63


def test_reference_lands_on_oracle_room_with_resets():
    from oracle.oracle import StructuredOracle
    steps, cap = 150, 30
    room = sc.room_scenario(steps=steps, range_sigma=5e-5)
    so, ref = StructuredOracle(cap), hp.HPFilter(cap)
    for s in range(steps):
        m = room["count"][s]
        z, R, u = room["z"][s, :m], room["R"][s, :m], room["u"][s]
        st, jo = so.scan(u, z, R)
        st2, jr = ref.scan(u, z, R)
        assert np.array_equal(jo, jr) and st == st2, "step %d" % s
        if s % 10 == 0 or s == steps - 1:
            _pin(so, ref, "room step %d" % s)
    assert so.stats()["resets"] > 0
    assert ref.min_margin >= 1e-6


def test_reference_lands_on_oracle_map_scenario():
    from oracle.oracle import StructuredOracle
    N, steps, m, cap = 60, 30, 8, 100
    scn = sc.map_scenario(N, steps, m=m, seed=21)
    so, ref = StructuredOracle(cap), hp.HPFilter(cap)
    so.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    ref.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    for s in range(steps):
        z = scn["z"][s].copy()
        if s % 7 == 3:
            z[-1, 1] += 3.0                       # a line that matches nothing: augmentation mid-run
        st, jo = so.scan(scn["u"][s], z, scn["R"][s])
        st2, jr = ref.scan(scn["u"][s], z, scn["R"][s])
        assert np.array_equal(jo, jr), "step %d" % s
    assert (jo >= 0).sum() >= m - 1
    _pin(so, ref, "map scenario")
    assert ref.min_margin >= 1e-6


def test_reference_lands_on_oracle_through_groups_and_a_reset():
    """The input generator of tests/test_gpu_pipeline_componentwise.py on a small map: ghosts appended and matched in
    the next scan, then a map reset and a rebuilt map that is re-observed.  The reference must agree with the
    structured oracle's associations at every scan, stay within the bound, and keep every gate decision at least 1e-6
    away from the threshold, so that the GPU cases rest on well-posed inputs."""
    import ctypes
    from oracle.oracle import StructuredOracle
    import test_gpu_pipeline_componentwise as pc
    c = pc.case_inputs("reset_small")
    so, ref = StructuredOracle(c["cap"], reset_headroom=c["headroom"]), hp.HPFilter(c["cap"], reset_headroom=c["headroom"])
    np.ctypeslib.as_array(so._lib.ekfo_y_ptr(so._h), shape=(so.n,))[:] = c["y"]
    so.P_view()[:] = c["P"]
    so._lib.ekfo_set_lines(so._h, ctypes.c_int(c["L"]))
    so.set_pose(c["y"][:3])
    ref.upload(c["y"], c["P"], c["L"])
    lines, matched_new = [], 0
    for s, (u, z, R) in enumerate(c["scans"]):
        L_before = ref.L
        st, jo = so.scan(u, z, R)
        st2, jr = ref.scan(u, z, R)
        assert np.array_equal(jo, jr) and st == st2, "scan %d: oracle %s, reference %s" % (s, jo, jr)
        assert so.lines == ref.L, "scan %d" % s
        if ref.L >= L_before and s:
            matched_new += int((jr >= lines[-1][0]).sum()) if lines[-1][1] > lines[-1][0] else 0
        lines.append((L_before, ref.L))
    assert sum(a < b for b, a in lines) == 1, lines                                          # one reset
    assert matched_new >= 8, "lines matched a landmark appended by the scan before: %d" % matched_new
    _pin(so, ref, "groups and a reset")
    assert ref.min_margin >= 1e-6


def test_componentwise_check_flags_sweep_faults_the_normwise_check_misses():
    """One scan of 8 matched lines on a 94-landmark map (nl = 191: the last 64-column tile is one short of full),
    P spread over 10 decades, the last landmarks' entries the smallest.  Faults applied to the reference's own result:
    one term missing on the last column, a term applied one column off, the last pending term of the pass dropped --
    each confined to the edge tile, as a sweep fault would be."""
    L, cap = 94, 100
    y, P, world = hp.spread_state(L, cap, 7, decades=(-6.0, -1.0))
    D = np.sqrt(np.diag(P)[3:3 + 2 * L])
    order = np.argsort(-D[::2])                    # landmarks by decreasing scale: put the smallest last
    y2, P2 = y.copy(), P.copy()
    idx = np.concatenate([[0, 1, 2], (3 + 2 * order[:, None] + np.arange(2)).ravel()])
    y2[:3 + 2 * L] = y[idx]; P2[:3 + 2 * L, :3 + 2 * L] = P[np.ix_(idx, idx)]
    world = world[order]
    ref = hp.HPFilter(cap, reset_headroom=0)
    ref.upload(y2, P2, L)
    rng = np.random.default_rng(3)
    z, R = hp.lines_for(world, hp.predicted_pose(tuple(y2[:3]), (0.02, 0.0, 0.01)), rng.choice(L - 20, 8, replace=False), rng)
    st, j = ref.scan((0.02, 0.0, 0.01), z, R)
    assert (j >= 0).all()
    _, _, Pv, Pm = ref.live()
    x = Pv.astype(np.float64)
    assert hp.worst_ratio(x, Pv, Pm) <= 1.0          # the reference rounded to doubles passes
    K, KS, _, _ = ref._terms()
    nl = ref.nl
    K = K[:nl].astype(np.float64); KS = KS[:nl].astype(np.float64)
    t = 64 * ((nl - 1) // 64)
    faults = {}
    f = x.copy()                                     # 1: term 0 missing on the last column of the edge tile
    f[t:, nl - 1] += KS[t:, 0] * K[nl - 1, 0] + KS[t:, 1] * K[nl - 1, 1]
    faults["term missing on the last column"] = f
    f = x.copy()                                     # 2: term 3 applied one column off inside the edge tile
    for c in range(t, nl - 1):
        f[t:, c] += KS[t:, 6:8] @ K[c, 6:8] - KS[t:, 6:8] @ K[c + 1, 6:8]
    faults["term one column off in the edge tile"] = f
    f = x.copy()                                     # 3: the last pending term dropped on the edge tile
    f[t:, t:] += KS[t:, -2:] @ K[t:, -2:].T
    faults["last pending term dropped"] = f
    passed_normwise = []
    for name, fx in faults.items():
        assert hp.worst_ratio(fx, Pv, Pm) > ref.C, name + ": not flagged by the componentwise check"
        if hp.normwise_ok(fx, Pv):
            passed_normwise.append(name)
    assert passed_normwise, "every fault was also visible normwise"
    print("faults the normwise 1e-9 check lets through:", passed_normwise)


# ---- ekf_gate_d2max (slam_ros_b200/csrc/ekf_internal.h) --------------------------------------------------------------
_GATE_MAIN = r"""
#include "ekf_internal.h"
#include <stdio.h>
#include <stdlib.h>
int main(int argc, char** argv) {
  for (int i = 1; i < argc; ++i) printf("%a\n", ekf_gate_d2max(strtod(argv[i], 0)));
  return 0;
}
"""


def _cuda_include():
    for d in (os.environ.get("CUDA_HOME", ""), "/usr/local/cuda"):
        if d and os.path.exists(os.path.join(d, "include", "cuda_runtime.h")):
            return os.path.join(d, "include")
    nvcc = shutil.which("nvcc")
    if nvcc:
        return os.path.join(os.path.dirname(os.path.dirname(nvcc)), "include")
    raise RuntimeError("CUDA headers not found (the library's build needs them too)")


def test_gate_threshold_function_returns_and_agrees_with_sqrt(tmp_path):
    """For every gate the function returns, and |d2| > T decides exactly as the reference's sqrt(|d2|) > gate.
    +inf used to spin for ever (nextafter(inf, inf) == inf)."""
    src = tmp_path / "gate.cpp"
    src.write_text(_GATE_MAIN)
    exe = tmp_path / "gate"
    subprocess.run(["g++", "-O1", "-std=c++17", "-I", os.path.join(ROOT, "slam_ros_b200", "csrc"), "-I", _cuda_include(),
                    str(src), "-o", str(exe)], check=True, capture_output=True, text=True)
    gates = [0.0, 1e-320, 0.4, 1e150, math.sqrt(1.7976931348623157e308), 1e200, math.inf, math.nan, -0.4]
    out = subprocess.run([str(exe)] + [g.hex() for g in gates], capture_output=True, text=True, timeout=30, check=True)
    Ts = [float.fromhex(s) for s in out.stdout.split()]
    assert len(Ts) == len(gates)
    rng = np.random.default_rng(5)
    for g, T in zip(gates, Ts):
        d2s = [0.0, -0.0, math.inf, -math.inf, math.nan]
        if math.isfinite(T):
            d2s += [math.nextafter(T, -math.inf), T, math.nextafter(T, math.inf), -T]
        d2s += list(10.0 ** rng.uniform(-300, 300, 200))
        if 0 < g < 1e150:
            d2s += list(g * g * np.exp(rng.uniform(-1e-3, 1e-3, 200)))
        for d2 in map(float, d2s):
            assert (abs(d2) > T) == (math.sqrt(abs(d2)) > g), (g, T, d2)
