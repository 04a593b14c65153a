"""CPU checks of the absolute pose fix (ekf_observe_pose) in the two references the GPU tests compare against.

Both are in tests/pose_fix_ref.py: the fix applied to the structured oracle's full matrix in float64, in the reference's
GSL pattern, and to the extended-precision reference (tests/hp_reference.py) in longdouble.

1. The oracle's fix against the extended-precision reference's,
   componentwise within C u mag, over a map scenario with fixes of every mask interleaved with scans, augmentation
   and a map reset.
2. The oracle against an independent closed form: for a full-pose fix P_rr' = (P_rr^-1 + R^-1)^-1 and
   P' = P - P H' S^-1 H P, in longdouble.
"""
import math

import numpy as np
import pytest

import hp_reference as hp
import pose_fix_ref as pf

LD = np.longdouble


def fix_R(rng, mask):
    """A full SPD 3x3 covariance with correlations (only the selected entries are read)."""
    A = rng.standard_normal((3, 3)) * np.array([0.02, 0.02, 0.01])[:, None]
    R = A @ A.T + np.diag([1e-4, 1e-4, 4e-5])
    return np.triu(R) + np.triu(R, 1).T


def noisy_pose(pose, rng):
    return np.asarray(pose) + rng.standard_normal(3) * np.array([0.01, 0.01, 0.005])


@pytest.fixture(scope="module")
def oracle_mod():
    from oracle import oracle as orc
    return orc


def test_pose_fix_oracle_against_hp_reference(oracle_mod):
    """60 landmarks in a filter of 90 (the reset fires once L > 80), 70 scans of 8 lines; a fix every third scan
    rotating through masks 1..7, from noisy true poses; ghost lines (3 m out) from scan 30 on append until the map
    resets, after which the map is rebuilt from the scans' lines."""
    from slam_ros_b200 import scenario as sc
    N, cap, S = 60, 90, 70
    scn = sc.map_scenario(N, S, m=8, seed=5)
    poses = sc.true_trajectory(scn["u"])
    o = oracle_mod.StructuredOracle(cap)
    ref = hp.HPFilter(cap)
    o.scan(np.zeros(3), scn["seed_z"], scn["seed_R"]); ref.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    rng = np.random.default_rng(7)
    masks, resets, appended, worst = [], 0, 0, 0.0
    for s in range(S):
        z = scn["z"][s].copy()
        if 30 <= s < 36:
            z[:, 1] += 3.0 + 0.5 * (s - 30)
        L0 = o.lines
        st, jo = o.scan(scn["u"][s], z, scn["R"][s])
        st_r, jr = ref.scan(scn["u"][s], z, scn["R"][s])
        assert np.array_equal(jo, jr), s
        assert o.lines == ref.L, s
        resets += o.lines < L0
        appended += int((jo < 0).sum())
        if s % 3 == 2:
            mask = 1 + len(masks) % 7
            masks.append(mask)
            zf, R = noisy_pose(poses[s + 1], rng), fix_R(rng, mask)
            so, d2o, So, vo = pf.oracle_observe_pose(o, zf, R, mask)
            sr, d2r = pf.hp_observe_pose(ref, zf, R, mask)
            assert so == sr == 1, (s, mask, so, sr)
            assert abs(d2o - d2r) <= 1e-9 * max(abs(d2r), 1.0), (s, d2o, d2r)
        y, P = o.live()
        yr, my, Pr, mP = ref.live()
        worst = max(worst, hp.check(y, yr, my, ref.C, "y, scan %d" % s) / ref.C)
        worst = max(worst, hp.check(P, Pr, mP, ref.C, "P, scan %d" % s) / ref.C)
        assert np.array_equal(o.pose, np.asarray(ref.pose, np.float64)) or \
            hp.worst_ratio(o.pose, ref.pose, ref.mpose) <= ref.C, s
    assert sorted(set(masks)) == list(range(1, 8))
    assert resets >= 1 and appended > 8 * 6
    assert worst <= 1.0


@pytest.mark.parametrize("mask", [1, 2, 3, 4, 5, 6, 7])
def test_pose_fix_oracle_against_closed_form(oracle_mod, mask):
    """P' = P - P H' S^-1 H P and y' = y + P H' S^-1 v in longdouble from the oracle's own state before the fix; for the
    full pose also the information form of the robot block, P_rr' = (P_rr^-1 + R^-1)^-1 (exact when H = [I 0])."""
    from slam_ros_b200 import scenario as sc
    N, cap = 40, 60
    scn = sc.map_scenario(N, 12, m=8, seed=13)
    o = oracle_mod.StructuredOracle(cap)
    o.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    for s in range(12):
        o.scan(scn["u"][s], scn["z"][s], scn["R"][s])
    rng = np.random.default_rng(mask)
    y0, P0 = o.live()
    sel = [c for c in range(3) if mask & (1 << c)]
    zf = y0[:3] + rng.standard_normal(3) * 0.01
    R = fix_R(rng, mask)
    st, d2, S, v = pf.oracle_observe_pose(o, zf, R, mask)
    assert st == 1
    y1, P1 = o.live()
    PL = P0.astype(LD)
    Ps = (PL + PL.T) / 2
    SL = Ps[np.ix_(sel, sel)] + R[np.ix_(sel, sel)].astype(LD)
    Si = np.linalg.inv(np.asarray(SL, np.float64)).astype(LD)
    for _ in range(3):
        Si = Si + Si @ (np.eye(len(sel), dtype=LD) - SL @ Si)
    vL = zf[sel].astype(LD) - y0[sel].astype(LD)
    for i, c in enumerate(sel):
        if c == 2:
            vL[i] = (vL[i] + LD(math.pi)) % LD(2 * math.pi) - LD(math.pi)
    G = Ps[:, sel] @ Si
    Pc = Ps - G @ Ps[sel, :]
    yc = y0.astype(LD) + G @ vL
    scale = float(np.abs(P0).max())
    assert float(np.abs(P1 - Pc).max()) <= 1e-12 * scale, float(np.abs(P1 - Pc).max()) / scale
    assert float(np.abs(y1[3:] - yc[3:]).max()) <= 1e-12 * max(float(np.abs(y0).max()), 1.0)
    assert float(np.abs(y1[:2] - yc[:2]).max()) <= 1e-12 * max(float(np.abs(y0).max()), 1.0)
    assert abs(float(d2) - float(vL @ Si @ vL)) <= 1e-9 * max(float(vL @ Si @ vL), 1.0)
    if mask == 7:
        Prr = Ps[:3, :3]
        info = np.linalg.inv(np.asarray(np.linalg.inv(np.asarray(Prr, np.float64)) + np.linalg.inv(R), np.float64))
        assert np.abs(P1[:3, :3] - info).max() <= 1e-9 * np.abs(info).max()


def test_pose_fix_oracle_gate_and_singular(oracle_mod):
    """d2_max = d2 accepts, the next double below rejects; theta alone on a fresh filter (P[2,2] = 0) with R_thth = 0
    is singular; neither a rejected nor a singular fix changes the oracle's state."""
    o = oracle_mod.StructuredOracle(20)
    y0, P0 = o.live()
    st, d2, S, v = pf.oracle_observe_pose(o, [0.0, 0.0, 0.3], np.zeros(9), 4)
    assert st == 2
    y1, P1 = o.live()
    assert np.array_equal(y0, y1) and np.array_equal(P0, P1)
    z, R = [0.05, -0.02, 0.0], np.diag([1e-3, 2e-3, 1e-3]).reshape(-1)
    st, d2, S, v = pf.oracle_observe_pose(o, z, R, 3, d2_max=0.0)
    assert st == 0 and d2 > 0
    assert np.array_equal(y0, o.live()[0]) and np.array_equal(P0, o.live()[1])
    assert pf.oracle_observe_pose(o, z, R, 3, d2_max=np.nextafter(d2, 0))[0] == 0
    assert pf.oracle_observe_pose(o, z, R, 3, d2_max=d2)[0] == 1
    assert not np.array_equal(P0, o.live()[1])
