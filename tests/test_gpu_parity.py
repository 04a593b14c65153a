"""GPU parity tests proper: libekfcuda (through its C ABI) against the CPU oracle on identical inputs.

Bar (BASELINE.json north_star): association indices bit-exact; state and P within 1e-9 relative after
every step, P measured as max|dP| / max|P| (the reference's P is not symmetric to the ulp, SURVEY Q12).
"""
import os

import numpy as np
import pytest

from slam_ros_b200 import scenario as sc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

TOL = 1e-9   # relative; north_star


def rel(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    den = max(np.abs(b).max(), 1e-300) if b.size else 1.0
    return float(np.abs(a - b).max() / den) if b.size else 0.0


def compare_state(f, so, ctx=""):
    y_o, P_o = so.live()
    y_g, P_g, L_g = f.download_live()
    assert L_g == so.lines, ctx + " line count"
    assert rel(y_g, y_o) < TOL, ctx + " y rel=%g" % rel(y_g, y_o)
    assert rel(P_g, P_o) < TOL, ctx + " P rel=%g" % rel(P_g, P_o)
    pose_g = f.pose
    assert rel(pose_g, so.pose) < TOL or np.abs(pose_g - so.pose).max() < 1e-12, ctx + " pose"


@pytest.fixture()
def oracle_cls():
    from oracle.oracle import StructuredOracle
    return StructuredOracle


def seed_pair(N, cap, oracle_cls, scn, **kw):
    from slam_ros_b200 import EkfFilter
    f = EkfFilter(capacity_lines=cap, **kw)
    so = oracle_cls(cap)
    rc, j, pose = f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    st, jo = so.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    assert rc == 0 and st == 0
    assert np.array_equal(j, jo)
    assert f.lines == so.lines == N
    return f, so


def test_create_initial_state(libekf, oracle_cls):
    from slam_ros_b200 import EkfFilter
    f = EkfFilter(capacity_lines=20)
    y, P, L = f.download()
    so = oracle_cls(20)
    assert L == 0 and np.array_equal(y, so.y_full()) and np.array_equal(P, so.P_full())
    assert P[0, 0] == 0.05 and P[1, 1] == 0.05


def test_seed_scan_augmentation(libekf, oracle_cls):
    scn = sc.map_scenario(40, 1, m=4, seed=3)
    f, so = seed_pair(40, 64, oracle_cls, scn)
    compare_state(f, so, "seed")
    # capacity layout download has zeros outside the live part
    y, P, L = f.download()
    nl = 3 + 2 * L
    assert np.all(P[nl:, :] == 0) and np.all(P[:, nl:] == 0) and np.all(y[nl:] == 0)
    assert np.array_equal(P, P.T)


def test_predict_only(libekf, oracle_cls):
    scn = sc.map_scenario(30, 5, m=4, seed=5)
    f, so = seed_pair(30, 40, oracle_cls, scn)
    for s in range(5):
        rc, j, pose = f.scan(scn["u"][s], np.zeros((0, 2)), np.zeros((0, 4)))
        so.scan(scn["u"][s], np.zeros((0, 2)), np.zeros((0, 4)))
        assert rc == 0
        compare_state(f, so, "predict %d" % s)


def test_stepwise_matches_oracle_primitives(libekf, oracle_cls):
    """ekf_predict / ekf_associate / ekf_update / ekf_add_line / ekf_end_scan one by one."""
    scn = sc.map_scenario(25, 6, m=5, seed=11)
    f, so = seed_pair(25, 40, oracle_cls, scn)
    for s in range(6):
        xg = f.predict(scn["u"][s])
        xo = so.predict(scn["u"][s])
        assert rel(xg, xo) < TOL
        n_lines = 0
        for i in range(scn["m"]):
            z, R = scn["z"][s, i], scn["R"][s, i]
            jg, innov_g = f.associate(z, R)
            jo, innov_o, d2 = so.associate(z, R)
            assert jg == jo, "step %d line %d" % (s, i)
            if jg >= 0:
                assert np.abs(innov_g - innov_o).max() < 1e-12
                f.update(jg, z, R)
                so.update(jo, z, R)
            else:
                f.add_line(z, R)
                so.queue(i)
            n_lines += 1
        rc, pose = f.end_scan(n_lines)
        st = so.end(scn["z"][s], scn["R"][s])
        assert rc == st == 0
        compare_state(f, so, "step-wise %d" % s)
    # independent full-scan replay for the state check
    f2, so2 = seed_pair(25, 40, oracle_cls, scn)
    for s in range(6):
        f2.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        so2.scan(scn["u"][s], scn["z"][s], scn["R"][s])
    compare_state(f2, so2, "fused replay")
    yg, Pg, Lg = f.download_live()
    y2, P2, L2 = f2.download_live()
    assert Lg == L2 and np.array_equal(yg, y2) and np.array_equal(Pg, P2), "step-wise path != fused path"


def test_gain_and_innovation_covariance(libekf, oracle_cls):
    scn = sc.map_scenario(16, 1, m=3, seed=21)
    f, so = seed_pair(16, 32, oracle_cls, scn)
    f.predict(scn["u"][0]); so.predict(scn["u"][0])
    z, R = scn["z"][0, 0], scn["R"][0, 0]
    jg, innov = f.associate(z, R)
    jo, innov_o, d2 = so.associate(z, R)
    assert jg == jo and jg >= 0
    f.update(jg, z, R); so.update(jo, z, R)
    rc, pose = f.end_scan(1)
    assert rc == 0
    so_y, so_P = so.live()
    yg, Pg, L = f.download_live()
    assert rel(Pg, so_P) < TOL and rel(yg, so_y) < TOL


@pytest.mark.parametrize("N,steps,m,seed", [(60, 300, 6, 1), (300, 200, 8, 2)])
def test_map_scenario_every_step(libekf, oracle_cls, N, steps, m, seed):
    scn = sc.map_scenario(N, steps, m=m, seed=seed)
    f, so = seed_pair(N, N + 96, oracle_cls, scn)
    for s in range(steps):
        rc, j, pose = f.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        st, jo = so.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        assert rc == st
        assert np.array_equal(j, jo), "association differs at step %d: %s vs %s" % (s, j, jo)
        if s % 10 == 0 or s == steps - 1:
            compare_state(f, so, "step %d" % s)
        else:
            assert rel(pose, so.pose) < TOL or np.abs(pose - so.pose).max() < 1e-12
    stats = so.stats()
    assert stats["matches"] > 0.8 * steps * m
    print("min gate margin |d - 0.4| = %.3e over %d gates" % (stats["min_margin"], stats["gates"]))


def test_all_launch_strategies_give_identical_bits(libekf):
    """Default (cluster line-loop kernel + TMA-pipelined sweep, each scan's sweep overlapped with the next
    scan's line loop on a second stream over a double-buffered P) vs the same without overlap, one rank-2
    sweep per match (reference-like), per-line kernels, the direct sweep kernel and forced mid-scan flushes."""
    from slam_ros_b200 import EkfFilter
    from slam_ros_b200.ekf import EKF_FLAG_EAGER_SWEEP, EKF_FLAG_SWEEP_DIRECT, EKF_FLAG_PER_LINE_KERNELS, EKF_FLAG_NO_OVERLAP
    scn = sc.map_scenario(80, 40, m=8, seed=9)
    variants = [EkfFilter(capacity_lines=128),                                  # overlapped two-stream pipeline
                EkfFilter(capacity_lines=128, flags=EKF_FLAG_NO_OVERLAP),
                EkfFilter(capacity_lines=128, flags=EKF_FLAG_EAGER_SWEEP),
                EkfFilter(capacity_lines=128, max_batch=3),                      # forces mid-scan flushes
                EkfFilter(capacity_lines=128, flags=EKF_FLAG_PER_LINE_KERNELS),
                EkfFilter(capacity_lines=128, flags=EKF_FLAG_SWEEP_DIRECT),
                EkfFilter(capacity_lines=128, flags=EKF_FLAG_PER_LINE_KERNELS | EKF_FLAG_SWEEP_DIRECT, max_batch=5)]
    for f in variants:
        f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    for s in range(40):
        outs = [f.scan(scn["u"][s], scn["z"][s], scn["R"][s]) for f in variants]
        for o in outs[1:]:
            assert np.array_equal(outs[0][1], o[1]) and np.array_equal(outs[0][2], o[2])
    ya, Pa, La = variants[0].download_live()
    for f in variants[1:]:
        y, P, L = f.download_live()
        assert L == La and np.array_equal(y, ya) and np.array_equal(P, Pa)


def test_room_scenario_with_resets(libekf, oracle_cls):
    """configs[0]: the reference-sized filter (LINESIZE=100) incl. augmentation, duplicates and map resets."""
    from slam_ros_b200 import EkfFilter
    steps = 400
    room = sc.room_scenario(steps=steps, range_sigma=5e-5)
    f = EkfFilter(capacity_lines=100)
    so = oracle_cls(100)
    for s in range(steps):
        m = room["count"][s]
        z, R, u = room["z"][s, :m], room["R"][s, :m], room["u"][s]
        rc, j, pose = f.scan(u, z, R)
        st, jo = so.scan(u, z, R)
        assert np.array_equal(j, jo), "step %d" % s
        assert f.lines == so.lines
        if s % 20 == 0 or s == steps - 1:
            compare_state(f, so, "room step %d" % s)
    assert so.stats()["resets"] > 0, "scenario should exercise the map reset"


def test_upload_download_roundtrip(libekf, oracle_cls):
    from slam_ros_b200 import EkfFilter
    scn = sc.map_scenario(20, 3, m=4, seed=4)
    f, so = seed_pair(20, 30, oracle_cls, scn)
    for s in range(3):
        f.scan(scn["u"][s], scn["z"][s], scn["R"][s])
    y, P, L = f.download()
    g = EkfFilter(capacity_lines=30)
    g.upload(y, P, L)
    y2, P2, L2 = g.download()
    assert L2 == L and np.array_equal(y, y2) and np.array_equal(P, P2)
    blk = f.download_block(2, 5, 7, 9)
    assert np.array_equal(blk, P[2:9, 5:14])
    tr, sm, sq = f.cov_stats()
    nl = 3 + 2 * L
    assert abs(tr - np.trace(P[:nl, :nl])) < 1e-12 * abs(tr)
    assert abs(sm - P.sum()) < 1e-9 * abs(P).sum()
    assert abs(sq - (P * P).sum()) < 1e-9 * (P * P).sum()
    assert np.array_equal(f.robot_cov(), P[:3, :3])


def test_capacity_policy(libekf, oracle_cls):
    """Q4: the reference overruns y[]; libekfcuda drops the lines that do not fit and reports it."""
    from slam_ros_b200 import EkfFilter
    from slam_ros_b200.ekf import EKF_ECAPACITY
    scn = sc.map_scenario(12, 1, m=2, seed=8)
    f = EkfFilter(capacity_lines=10, reset_headroom=0)
    so = oracle_cls(10, reset_headroom=0)
    rc, j, pose = f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    st, jo = so.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    assert rc == EKF_ECAPACITY and st == 2
    assert f.lines == so.lines == 10
    compare_state(f, so, "capacity")


def test_sweep_probe_leaves_state_bitwise(libekf, oracle_cls):
    scn = sc.map_scenario(200, 2, m=8, seed=6)
    f, so = seed_pair(200, 256, oracle_cls, scn)
    f.scan(scn["u"][0], scn["z"][0], scn["R"][0])
    y0, P0, L0 = f.download_live()
    for m in (1, 2, 4, 8, 13):
        ms = f.sweep_probe(m=m, repeats=3)
        assert ms > 0
    y1, P1, L1 = f.download_live()
    assert np.array_equal(P0, P1) and np.array_equal(y0, y1)


def test_ellipse_matches_oracle(libekf, oracle_cls):
    scn = sc.map_scenario(10, 4, m=3, seed=2)
    f, so = seed_pair(10, 20, oracle_cls, scn)
    for s in range(4):
        f.scan(scn["u"][s], scn["z"][s], scn["R"][s]); so.scan(scn["u"][s], scn["z"][s], scn["R"][s])
    okg, axg, ang = f.get_ellipse()
    oko, axo, ano = so.get_ellipse()
    assert okg and oko
    assert np.allclose(axg, axo, rtol=1e-6) and abs(ang - ano) < 1e-5


def test_robot_mirror_against_literal_reference(libekf):
    """The host-side `Robot` mirror driven exactly like the reference's node drives Robot::localize."""
    from oracle.oracle import LiteralReference, have_literal
    if not have_literal():
        pytest.skip("oracle/_ref/libslamref.so not present")
    from slam_ros_b200 import Robot, Line
    lit = LiteralReference()
    rb = Robot(0, 0, 0)
    steps = 120
    room = sc.room_scenario(steps=steps, range_sigma=5e-5)
    for s in range(steps):
        m = room["count"][s]
        z, R, u = room["z"][s, :m], room["R"][s, :m], room["u"][s]
        y_l, P_l, L_l, pose_l = lit.state()
        enc_l = sc.encoder_for(pose_l, u)
        enc_g = sc.encoder_for((rb.xPos, rb.yPos, rb.thetaPos), u)
        lit.localize(z, R, enc_l)
        rb.localize([Line(z[i, 0], z[i, 1], R[i]) for i in range(m)], rot=None, encoder=enc_g)
        y_l, P_l, L_l, pose_l = lit.state()
        assert rb.savedLineCount == L_l, "step %d" % s
        assert np.abs(np.array([rb.xPos, rb.yPos, rb.thetaPos]) - pose_l).max() < 1e-9
    assert rel(rb.P_t0, P_l) < TOL and rel(rb.y, y_l) < TOL


def test_robot_mirror_against_golden_vectors_of_the_reference(libekf):
    """The same drive on the outputs the reference's own Robot.cpp produced (tests/golden/room_literal.npz, made by
    make_golden.py): the fixture's lines and odometry u, savedLineCount and the pose after every step, y and P_t0 where
    the fixture kept them, the ellipse at the end.  As in the live test, the encoder pose is the one that makes
    Robot.cpp:140-145 recover u from the mirror's OWN pose: the fixture's encoder poses would turn the last bits in
    which two poses differ into a difference of odometry (u[2] = theta - encoder[2]), compounding step after step."""
    from slam_ros_b200 import Robot, Line
    g = np.load(os.path.join(ROOT, "tests", "golden", "room_literal.npz"))
    rb = Robot(0, 0, 0)
    for s in range(g["u"].shape[0]):
        m = int(g["count"][s])
        z, R = g["z"][s, :m], g["R"][s, :m]
        enc = sc.encoder_for((rb.xPos, rb.yPos, rb.thetaPos), g["u"][s])
        rb.localize([Line(z[i, 0], z[i, 1], R[i]) for i in range(m)], rot=None, encoder=enc)
        assert rb.savedLineCount == int(g["L"][s]), "step %d" % s
        assert np.abs(np.array([rb.xPos, rb.yPos, rb.thetaPos]) - g["pose"][s]).max() < 1e-9, "pose at step %d" % s
        if ("P_%d" % s) in g.files:
            assert rel(rb.P_t0, g["P_%d" % s]) < TOL and rel(rb.y, g["y_%d" % s]) < TOL, "state at step %d" % s
    ok, ax, ang = rb.getEllipse()
    assert ok and np.allclose(ax, g["ellipse"][:2], rtol=1e-5) and abs(ang - g["ellipse"][2]) < 1e-4


def test_batch_filters_match_oracle(libekf, oracle_cls):
    from slam_ros_b200 import EkfBatch
    B, N, m, steps = 6, 12, 4, 25
    scns = [sc.map_scenario(N, steps, m=m, seed=100 + f) for f in range(B)]
    cap = 24
    bt = EkfBatch(B, capacity_lines=cap)
    sos = [oracle_cls(cap) for _ in range(B)]
    rc, j, pose = bt.scan(np.zeros((B, 3)), np.stack([s["seed_z"] for s in scns]), np.stack([s["seed_R"] for s in scns]))
    for f in range(B):
        sos[f].scan(np.zeros(3), scns[f]["seed_z"], scns[f]["seed_R"])
    for s in range(steps):
        rc, j, pose = bt.scan(np.stack([x["u"][s] for x in scns]), np.stack([x["z"][s] for x in scns]),
                              np.stack([x["R"][s] for x in scns]))
        for f in range(B):
            st, jo = sos[f].scan(scns[f]["u"][s], scns[f]["z"][s], scns[f]["R"][s])
            assert np.array_equal(j[f], jo), "filter %d step %d" % (f, s)
            assert np.abs(pose[f] - sos[f].pose).max() < 1e-10
    for f in range(B):
        y, P, L, pose_f = bt.download(f)
        assert L == sos[f].lines
        assert rel(y, sos[f].y_full()) < TOL and rel(P, sos[f].P_full()) < TOL


def test_large_map_properties(libekf, oracle_cls):
    """Full-size style checks that do not need the oracle at full size: symmetry of the read-out, trace
    never increases through an update, eager == deferred on a 2k-landmark map, spot blocks against the
    oracle on a short prefix."""
    N, steps, m = 2000, 6, 8
    scn = sc.map_scenario(N, steps, m=m, seed=77)
    f, so = seed_pair(N, N + 64, oracle_cls, scn)
    tr_prev = None
    for s in range(steps):
        rc, j, pose = f.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        st, jo = so.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        assert np.array_equal(j, jo)
    y_o, P_o = so.live()
    for (r0, c0) in ((0, 0), (3, 3), (1000, 17), (17, 1000), (3900, 3900), (2047, 63), (64, 2048)):
        nr = min(70, P_o.shape[0] - r0); nc = min(70, P_o.shape[1] - c0)
        blk = f.download_block(r0, c0, nr, nc)
        ref = P_o[r0:r0 + nr, c0:c0 + nc]
        assert np.abs(blk - ref).max() / np.abs(P_o).max() < TOL, (r0, c0)
    tr, sm, sq = f.cov_stats()
    assert abs(tr - np.trace(P_o)) / abs(np.trace(P_o)) < TOL
    assert abs(sq - (P_o * P_o).sum()) / (P_o * P_o).sum() < 1e-8


def test_thousand_steps_every_step(libekf, oracle_cls):
    """north_star: association bit-exact and state/P within 1e-9 relative after EACH step over 1k steps."""
    N, steps, m = 120, 1000, 8
    scn = sc.map_scenario(N, steps, m=m, seed=31)
    f, so = seed_pair(N, N + 400, oracle_cls, scn)
    worst_y = worst_P = 0.0
    for s in range(steps):
        rc, j, pose = f.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        st, jo = so.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        assert rc == st
        assert np.array_equal(j, jo), "association differs at step %d" % s
        y_o, P_o = so.live()
        y_g, P_g, L_g = f.download_live()
        assert L_g == so.lines
        worst_y = max(worst_y, rel(y_g, y_o)); worst_P = max(worst_P, rel(P_g, P_o))
        assert worst_y < TOL and worst_P < TOL, "step %d: y %.2e P %.2e" % (s, worst_y, worst_P)
    st = so.stats()
    print("1000 steps: worst rel err y %.2e, P %.2e; min gate margin %.3e over %d gates; %d matches"
          % (worst_y, worst_P, st["min_margin"], st["gates"], st["matches"]))


@pytest.mark.parametrize("m", [32, 64])
def test_batched_multi_line_updates(libekf, oracle_cls, m):
    """configs[2]: m = 32 / 64 observed lines per step folded into one deferred rank-2m sweep."""
    N, steps = 700, 6
    scn = sc.map_scenario(N, steps, m=m, seed=50 + m, stride=m + 3)
    f, so = seed_pair(N, N + 128, oracle_cls, scn)
    for s in range(steps):
        rc, j, pose = f.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        st, jo = so.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        assert np.array_equal(j, jo), "step %d" % s
        compare_state(f, so, "m=%d step %d" % (m, s))
    assert so.stats()["matches"] > 0.8 * steps * m


@pytest.mark.parametrize("m", [16, 32, 40, 64])
def test_overlapped_pipeline_with_large_line_groups(libekf, oracle_cls, m):
    """m = 16 / 32 lines per scan on a map large enough (n = 6203) for the overlapped path: the scan's 16 / 32
    pending terms are folded by ONE out-of-place sweep pass (16- / 32-term template) while the next scan's line loop
    corrects its column reads with up to 2m pending terms.  m = 40 / 64: the scan goes through the pipeline as chunks
    of 16 lines (16 + 16 + 8 / 4 x 16), each chunk's sweep under the next chunk's line loop; two of those scans carry
    lines that match nothing, so the map grows at the end of a chunked scan.  Checked against the oracle and, bit for
    bit, against the non-overlapped in-place path."""
    from slam_ros_b200 import EkfFilter
    from slam_ros_b200.ekf import EKF_FLAG_NO_OVERLAP
    N, steps = 3100, 7
    scn = sc.map_scenario(N, steps, m=m, seed=70 + m, stride=m + 3)
    if m > 32:
        for s, lines in ((2, (5, 20, 37)), (4, (0, 17, m - 1))):
            for i in lines:
                scn["z"][s][i, 1] += 3.0 + 0.1 * i
    f, so = seed_pair(N, N + 128, oracle_cls, scn)
    so._lib.ekfo_set_threads(so._h, 0)
    g = EkfFilter(capacity_lines=N + 128, flags=EKF_FLAG_NO_OVERLAP)
    g.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    for s in range(steps):
        rc, j, pose = f.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        rg, jg, pg = g.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        st, jo = so.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        assert np.array_equal(j, jo) and np.array_equal(jg, jo), "step %d" % s
        assert np.array_equal(pose, pg)
        if s in (2, steps - 1):
            compare_state(f, so, "m=%d step %d" % (m, s))
    assert so.stats()["matches"] > 0.8 * steps * m
    yf, Pf, Lf = f.download_live()
    yg, Pg, Lg = g.download_live()
    assert Lf == Lg and np.array_equal(yf, yg) and np.array_equal(Pf, Pg)
    if m > 32:
        assert Lf == N + 6


def test_empty_and_ragged_scans(libekf, oracle_cls):
    """Edge cases: scans with no lines, one line, lines on an empty map, duplicated observations of one landmark."""
    from slam_ros_b200 import EkfFilter
    scn = sc.map_scenario(20, 8, m=6, seed=13)
    f = EkfFilter(capacity_lines=64); so = oracle_cls(64)
    for o in (0, 1):                                   # empty map, empty scan
        rc, j, pose = f.scan(scn["u"][0], np.zeros((0, 2)), np.zeros((0, 4)))
        so.scan(scn["u"][0], np.zeros((0, 2)), np.zeros((0, 4)))
    compare_state(f, so, "empty")
    rc, j, pose = f.scan(np.zeros(3), scn["seed_z"][:1], scn["seed_R"][:1])       # a single line on the empty map
    so.scan(np.zeros(3), scn["seed_z"][:1], scn["seed_R"][:1])
    rc, j, pose = f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])               # the first line now matches landmark 0
    st, jo = so.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    assert np.array_equal(j, jo) and j[0] == 0
    compare_state(f, so, "seed after single")
    for s in range(8):
        k = s % 5 + 1
        z = np.concatenate([scn["z"][s, :k], scn["z"][s, :1]])                     # ragged + a duplicated observation
        R = np.concatenate([scn["R"][s, :k], scn["R"][s, :1]])
        rc, j, pose = f.scan(scn["u"][s], z, R)
        st, jo = so.scan(scn["u"][s], z, R)
        assert np.array_equal(j, jo), "step %d" % s
    compare_state(f, so, "ragged")


def test_full_size_10k_landmarks_against_oracle(libekf, oracle_cls):
    """BASELINE.json configs[2] at full size (P 20003^2 fp64 = 3.2 GB): a short prefix against the oracle
    (association bit-exact; y exactly comparable; P compared on blocks spread over the matrix and through the
    size-independent invariants trace / sum of squares), then invariants over more steps: the trace never
    grows through an update scan beyond what prediction adds, and the read-out stays symmetric."""
    N, steps, m = 10000, 4, 8
    scn = sc.map_scenario(N, 12, m=m, seed=1)
    f, so = seed_pair(N, N + 256, oracle_cls, scn, )
    so._lib.ekfo_set_threads(so._h, 0)          # all host threads for the n^2 sweeps of the checker
    for s in range(steps):
        rc, j, pose = f.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        st, jo = so.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        assert rc == st == 0 and np.array_equal(j, jo), "step %d" % s
    nl = 3 + 2 * so.lines
    Pv = so.P_view()
    pmax = float(np.abs(Pv[:nl, :nl]).max())
    y_g = f.download_y()
    assert rel(y_g, so.y_full()[:nl]) < TOL
    rng = np.random.default_rng(0)
    corners = [(0, 0), (0, nl - 80), (nl - 80, nl - 80), (3, 3)] + [tuple(rng.integers(0, nl - 80, 2)) for _ in range(12)]
    for (r0, c0) in corners:
        blk = f.download_block(int(r0), int(c0), 80, 80)
        ref = Pv[r0:r0 + 80, c0:c0 + 80]
        assert np.abs(blk - ref).max() / pmax < TOL, (r0, c0)
        blk_t = f.download_block(int(c0), int(r0), 80, 80)
        assert np.array_equal(blk, blk_t.T)                       # symmetric read-out
    tr, sm, sq = f.cov_stats()
    tr_o = float(np.trace(Pv[:nl, :nl]))
    assert abs(tr - tr_o) / abs(tr_o) < TOL
    sq_o = float(np.einsum("ij,ij->", Pv[:nl, :nl], Pv[:nl, :nl]))
    assert abs(sq - sq_o) / sq_o < 1e-8
    for s in range(steps, 12):                                     # invariants only (no CPU sweep)
        tr_before = f.cov_stats()[0]
        rc, j, pose = f.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        tr_after = f.cov_stats()[0]
        assert rc == 0 and (j >= 0).sum() >= m - 2
        assert tr_after < tr_before + 1e-2                         # prediction adds <= 4q ~ 2e-3; updates only remove


def test_chunked_scan_through_capacity_map_reset_and_empty_map(libekf, oracle_cls):
    """A chunked (40-line) scan whose unmatched lines take the map beyond capacity - headroom: the map is reset at the end
    of the scan while the sweeps of its earlier chunks may still be in flight; the next 40-line scan then meets an EMPTY
    map (every line queued, no chunking, the in-place path), the one after a 40-landmark map, and a 100-line scan (more
    than the 64 lines the tables start with) grows the tables.  Every step against the oracle."""
    N, m = 3100, 40
    scn = sc.map_scenario(N, 5, m=m, seed=91, stride=m + 3)
    f, so = seed_pair(N, N + 20, oracle_cls, scn)
    so._lib.ekfo_set_threads(so._h, 0)
    wide = sc.map_scenario(N, 1, m=100, seed=92, stride=7)
    for s in range(5):
        z, R = scn["z"][s].copy(), scn["R"][s].copy()
        if s == 1:
            z[::3, 1] += 5.0 + 0.05 * np.arange(z[::3].shape[0])    # 14 lines match nothing: L = N + 14 > capacity - 10
        if s == 4:
            z, R = wide["z"][0].copy(), wide["R"][0].copy()          # 100 lines on a small map
        rc, j, pose = f.scan(scn["u"][s], z, R)
        st, jo = so.scan(scn["u"][s], z, R)
        assert rc == st and np.array_equal(j, jo), "step %d" % s
        assert f.lines == so.lines, "step %d" % s
        if s == 0:
            compare_state(f, so, "before the reset")
    assert so.stats()["resets"] == 1 and so.lines > 40
    compare_state(f, so, "after reset, empty map and table growth")


@pytest.mark.parametrize("N,cap_extra,m", [(3100, 128, 8), (10200, 560, 8), (10200, 560, 32)])
def test_device_resident_scans_equal_the_host_path(libekf, N, cap_extra, m):
    """ekf_scan_device (inputs already in HBM, no read-back: the path bench.py's `value` times) against ekf_scan on the same
    sequence, bit for bit: a burst the host never waits for (its bound of the map size only drifts upwards, past the
    threads of the register-resident line loop at 10 200 landmarks), then paced scans with a pause in between (the
    asynchronous snapshot of the device state lands and tightens the bound), with lines that match nothing so that the
    map really grows, then a burst again."""
    import time
    import torch
    from slam_ros_b200 import EkfFilter
    steps = 36
    scn = sc.map_scenario(N, steps, m=m, seed=17, stride=m + 3)
    for s in (3, 9, 20, 21, 30):
        scn["z"][s][1, 1] += 6.0 + 0.01 * s                         # one new landmark in each of these scans
    f = EkfFilter(capacity_lines=N + cap_extra)                     # device-resident inputs
    g = EkfFilter(capacity_lines=N + cap_extra)                     # host buffers
    for x in (f, g):
        x.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    dev = torch.device("cuda:0")
    d_u = torch.tensor(scn["u"], dtype=torch.float64, device=dev)
    d_z = torch.tensor(scn["z"], dtype=torch.float64, device=dev)
    d_R = torch.tensor(scn["R"], dtype=torch.float64, device=dev)
    d_j = torch.full((steps, m), -7, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    for s in range(steps):
        f.scan_device(d_u[s].data_ptr(), m, d_z[s].data_ptr(), d_R[s].data_ptr(), d_j[s].data_ptr())
        if 12 <= s < 24:
            time.sleep(0.02)                                        # paced: the snapshots land
    f.sync()
    j_dev = d_j.cpu().numpy()
    for s in range(steps):
        rc, j, pose = g.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        assert rc == 0 and np.array_equal(j, j_dev[s]), "step %d" % s
    assert f.lines == g.lines == N + 5
    assert np.array_equal(f.pose, g.pose) and f.cov_stats() == g.cov_stats()
    assert np.array_equal(f.download_y(), g.download_y())
    nl = 3 + 2 * g.lines
    for (r0, c0) in [(0, 0), (0, nl - 64), (nl - 64, nl - 64), (1000, 5000)]:
        assert np.array_equal(f.download_block(r0, c0, 64, 64), g.download_block(r0, c0, 64, 64)), (r0, c0)


def test_overlapped_pipeline_with_changing_line_counts(libekf):
    """Scans of 8 / 32 / 64 / 16 / 40 lines in turn on a map whose capacity (10 752 lines) makes the line loop of the
    longer scans take 21 SMs instead of 20 (one thread per landmark of the capacity): the sweep in flight was sized for
    the previous scan's class, so a wider line loop first waits for it.  Bit for bit against the in-place path."""
    from slam_ros_b200 import EkfFilter
    from slam_ros_b200.ekf import EKF_FLAG_NO_OVERLAP
    N = 10400
    ms = [8, 32, 8, 64, 16, 8, 40, 8]
    scn = sc.map_scenario(N, len(ms), m=64, seed=5, stride=67)
    f = EkfFilter(capacity_lines=N + 352)
    g = EkfFilter(capacity_lines=N + 352, flags=EKF_FLAG_NO_OVERLAP)
    for x in (f, g):
        x.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    for s, m in enumerate(ms):
        z, R = scn["z"][s][:m].copy(), scn["R"][s][:m].copy()
        if s == 3:
            z[11, 1] += 4.0                                         # one line of the chunked scan matches nothing
        rc, j, pose = f.scan(scn["u"][s], z, R)
        rg, jg, pg = g.scan(scn["u"][s], z, R)
        assert rc == rg == 0 and np.array_equal(j, jg) and np.array_equal(pose, pg), "step %d" % s
        assert (j >= 0).sum() >= m - 2
    assert f.cov_stats() == g.cov_stats()
    assert np.array_equal(f.download_y(), g.download_y())
    nl = 3 + 2 * (N + 1)
    for (r0, c0) in [(0, 0), (0, nl - 80), (nl - 80, nl - 80), (5000, 9000), (123, 20000)]:
        assert np.array_equal(f.download_block(r0, c0, 80, 80), g.download_block(r0, c0, 80, 80)), (r0, c0)


def test_overlapped_pipeline_interleaved_with_stepwise_calls(libekf, oracle_cls):
    """A map large enough (n = 6203) for the overlapped two-stream path, with fused scans, step-wise scans,
    downloads and sweep probes interleaved: every switch drains the sweep in flight."""
    N, steps, m = 3100, 14, 8
    scn = sc.map_scenario(N, steps, m=m, seed=23)
    f, so = seed_pair(N, N + 64, oracle_cls, scn)
    so._lib.ekfo_set_threads(so._h, 0)
    for s in range(steps):
        z, R, u = scn["z"][s], scn["R"][s], scn["u"][s]
        if s % 4 == 2:                                   # step-wise scan in the middle of overlapped ones
            f.predict(u); so.predict(u)
            for i in range(m):
                jg, _ = f.associate(z[i], R[i]); jo, _, _ = so.associate(z[i], R[i])
                assert jg == jo
                if jg >= 0:
                    f.update(jg, z[i], R[i]); so.update(jo, z[i], R[i])
                else:
                    f.add_line(z[i], R[i]); so.queue(i)
            rc, pose = f.end_scan(m); so.end(z, R)
        else:
            rc, j, pose = f.scan(u, z, R)
            st, jo = so.scan(u, z, R)
            assert np.array_equal(j, jo), "step %d" % s
        if s % 5 == 4:
            f.sweep_probe(m=3, repeats=1)               # forces a drain; must leave the state untouched
            compare_state(f, so, "interleaved step %d" % s)
    compare_state(f, so, "interleaved final")


def test_line_loop_forms_give_identical_bits(libekf):
    """The one-barrier line loop (k_scan_lines2: a thread owns its landmarks' hot entries AND gain rows) against the
    first two-barrier form (EKF_LINE_LOOP=1): cluster launch on a small map, cooperative launch beside the overlapped
    sweep on a large one, more landmarks than threads (several landmarks per thread: hot entries from memory), scans with
    unmatched lines (augmentation) in between -- matches, state and covariance bit for bit."""
    import subprocess
    import sys
    code = (
        "import sys, numpy as np\n"
        "sys.path.insert(0, %r)\n"
        "from slam_ros_b200 import EkfFilter, scenario as sc\n"
        "out = {}\n"
        "for N, m, steps in ((700, 8, 12), (3300, 8, 10), (3300, 24, 6), (12000, 8, 4)):\n"
        "    scn = sc.map_scenario(N, steps, m=m, seed=5)\n"
        "    f = EkfFilter(capacity_lines=N + 96)\n"
        "    f.scan(np.zeros(3), scn['seed_z'], scn['seed_R'])\n"
        "    J = []\n"
        "    for s in range(steps):\n"
        "        z = scn['z'][s].copy()\n"
        "        if s %% 4 == 2: z[1::2, 1] += 3.0\n"
        "        J.append(f.scan(scn['u'][s], z, scn['R'][s])[1])\n"
        "    y = f.download_y()\n"
        "    k = '%%d_%%d' %% (N, m)\n"
        "    out['J_' + k] = np.stack(J); out['y_' + k] = y\n"
        "    out['B_' + k] = np.stack([f.download_block(r0, c0, 64, 64) for r0, c0 in ((0, 0), (3, 3), (5, 900), (700, 1100), (len(y) - 64, len(y) - 64))])\n"
        "    out['S_' + k] = np.array(f.cov_stats())\n"
        "    f.close()\n"
        "np.savez(sys.argv[1], **out)\n"
    ) % ROOT
    res = []
    for v in ("1", "0"):
        path = "/tmp/ekf_lineloop_%s_%d.npz" % (v, os.getpid())
        env = dict(os.environ, EKF_LINE_LOOP=v)
        out = subprocess.run([sys.executable, "-c", code, path], capture_output=True, text=True, timeout=900, env=env)
        assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
        res.append(dict(np.load(path)))
        os.remove(path)
    for k in res[0]:
        assert np.array_equal(res[0][k], res[1][k]), k
    assert (res[0]["J_700_8"] >= 0).sum() > 50 and (res[0]["J_700_8"] < 0).sum() > 5


@pytest.mark.parametrize("shape", [0, 9, 10])
def test_sweep_kernels_give_identical_bits(libekf, shape):
    """EKF_SWEEP_SHAPE selects the consumers of the pipelined sweep: 11 = k_sweep_quad for every count (8x4 register
    tiles, DFMA), 0 = the default (quad up to 8 pending terms, tensor cores beyond), 9 = k_sweep_pipe (8x2),
    10 = k_sweep_dmma for every count (fp64 tensor cores: mma.sync.m8n8k4.f64 accumulates as the k-ordered FMA chain,
    i.e. sub_rank2 term after term -- measured, scripts/dmma_probe.cu).  Same scans, m = 8 / 13 / 32 / 40 lines (odd
    counts: the tensor-core step's zero-padded second term; > 32: two passes): the downloaded state must equal the
    all-DFMA run's bit for bit, and the oracle's within 1e-9."""
    import subprocess
    import sys
    code = (
        "import sys, numpy as np\n"
        "sys.path.insert(0, %r)\n"
        "from slam_ros_b200 import EkfFilter, scenario as sc\n"
        "out = {}\n"
        "for N, m in ((700, 8), (700, 13), (3300, 32), (3300, 40)):\n"
        "    scn = sc.map_scenario(N, 5, m=m, seed=3)\n"
        "    f = EkfFilter(capacity_lines=N + 96)\n"
        "    f.scan(np.zeros(3), scn['seed_z'], scn['seed_R'])\n"
        "    J = [f.scan(scn['u'][s], scn['z'][s], scn['R'][s])[1] for s in range(5)]\n"
        "    y, P, L = f.download_live()\n"
        "    out['J_%%d_%%d' %% (N, m)] = np.stack(J); out['y_%%d_%%d' %% (N, m)] = y; out['P_%%d_%%d' %% (N, m)] = P\n"
        "    f.close()\n"
        "np.savez(sys.argv[1], **out)\n"
    ) % ROOT
    res = []
    for sh in (11, shape):
        path = "/tmp/ekf_shape_%d_%d.npz" % (sh, os.getpid())
        env = dict(os.environ, EKF_SWEEP_SHAPE=str(sh))
        out = subprocess.run([sys.executable, "-c", code, path], capture_output=True, text=True, timeout=600, env=env)
        assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
        res.append(dict(np.load(path)))
        os.remove(path)
    for k in res[0]:
        assert np.array_equal(res[0][k], res[1][k]), k
    # and against the oracle, for the largest case
    from oracle.oracle import StructuredOracle
    N, m = 3300, 40
    scn = sc.map_scenario(N, 5, m=m, seed=3)
    so = StructuredOracle(N + 96, threads=0)
    so.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    Jo = np.stack([so.scan(scn["u"][s], scn["z"][s], scn["R"][s])[1] for s in range(5)])
    yo, Po = so.live()
    assert np.array_equal(res[1]["J_3300_40"], Jo)
    assert rel(res[1]["P_3300_40"], Po) < TOL and rel(res[1]["y_3300_40"], yo) < TOL


@pytest.mark.parametrize("maxc", [8, 16, 32])
def test_sweep_ring_for_every_pending_count_and_pass_width(libekf, maxc):
    """The stand-alone sweep for every pending-term count 1..64 and every pass width (EKF_SWEEP_MAXC), state
    untouched bit for bit.  Regression: with a 3-stage ring shared by the two consumer groups, a group that ran
    ahead mistook the other group's tile for its own (mbarrier waits only see a phase parity) -- found as a launch
    failure at 17 terms with 16-term passes; each (stage, group) now has its own full barrier."""
    import subprocess
    import sys
    code = (
        "import sys, numpy as np\n"
        "sys.path.insert(0, %r)\n"
        "from slam_ros_b200 import EkfFilter, scenario as sc\n"
        "N = 1500\n"
        "scn = sc.map_scenario(N, 1, m=8, seed=1)\n"
        "f = EkfFilter(capacity_lines=N + 64)\n"
        "f.scan(np.zeros(3), scn['seed_z'], scn['seed_R'])\n"
        "s0 = f.cov_stats()\n"
        "for mm in range(1, 65):\n"
        "    f.sweep_probe(m=mm, repeats=2)\n"
        "assert f.cov_stats() == s0\n"
        "print('all counts ok')\n"
    ) % ROOT
    env = dict(os.environ, EKF_SWEEP_MAXC=str(maxc))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0 and "all counts ok" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


def test_overlapped_pipeline_through_augmentation_capacity_and_map_reset(libekf, oracle_cls):
    """The overlapped two-stream path (n = 6203) while the map GROWS (unmatched lines appended while the previous
    scan's sweep is in flight), hits the capacity policy (Q4: lines that do not fit are dropped, EKF_ECAPACITY) and
    the map reset (Robot.cpp:893-904: savedLineCount > capacity - headroom wipes the map), then rebuilds -- all
    without leaving the asynchronous path; every step's matches and pose against the oracle, state at the end."""
    from slam_ros_b200.ekf import EKF_ECAPACITY
    N, steps, m = 3100, 12, 8
    scn = sc.map_scenario(N, steps, m=m, seed=61)
    cap = N + 14                                              # reset when L > cap - 10 = 3104; room for 14 new lines
    f, so = seed_pair(N, cap, oracle_cls, scn)
    so._lib.ekfo_set_threads(so._h, 0)
    rng = np.random.default_rng(5)
    saw_capacity = saw_reset = False
    for s in range(steps):
        z = scn["z"][s].copy(); R = scn["R"][s].copy()
        if s >= 2:                                            # half of the lines are walls the map has never seen
            z[4:, 0] = rng.uniform(-3.0, 3.0, m - 4)
            z[4:, 1] = rng.uniform(20.0, 30.0, m - 4)
        L_before = so.lines
        rc, j, pose = f.scan(scn["u"][s], z, R)
        st, jo = so.scan(scn["u"][s], z, R)
        assert np.array_equal(j, jo), "step %d: %s vs %s" % (s, j, jo)
        assert rel(pose, so.pose) < TOL or np.abs(pose - so.pose).max() < 1e-12
        assert rc == st
        saw_capacity |= (rc == EKF_ECAPACITY)
        saw_reset |= (so.lines < L_before)
        if s in (3, 6, steps - 1):
            compare_state(f, so, "step %d" % s)
    assert saw_reset, "the scenario must drive the map through a reset"
    assert f.state()[1] == so.lines


def test_overlapped_pipeline_with_ragged_scans(libekf, oracle_cls):
    """Scans of 8, 0, 3, 16, 40, 1, 32, 8, 33, 2 lines on a map large enough for the overlapped path: empty scans,
    group sizes that select the 8- / 16- / 32-term sweep, and scans above 32 lines that drain the pipeline and run
    synchronously, back to back."""
    N = 3100
    ms = [8, 0, 3, 16, 40, 1, 32, 8, 33, 2]
    scn = sc.map_scenario(N, len(ms), m=40, seed=77, stride=43)
    f, so = seed_pair(N, N + 64, oracle_cls, scn)
    so._lib.ekfo_set_threads(so._h, 0)
    for s, m in enumerate(ms):
        z, R = scn["z"][s, :m], scn["R"][s, :m]
        rc, j, pose = f.scan(scn["u"][s], z, R)
        st, jo = so.scan(scn["u"][s], z, R)
        assert rc == st and np.array_equal(j, jo), "step %d (m = %d)" % (s, m)
        assert rel(pose, so.pose) < TOL or np.abs(pose - so.pose).max() < 1e-12
        if s in (4, 7, len(ms) - 1):
            compare_state(f, so, "step %d" % s)


def test_against_golden_vectors_of_the_reference_at_linesize_1000(libekf):
    """tests/golden/literal_1k.npz was produced by the reference's OWN Robot.cpp compiled with LINESIZE = 1000
    (BASELINE configs[1] size; make_golden_1k.py).  libekfcuda, fed the same inputs through the Robot mirror's
    arithmetic (pose - encoder odometry), must land on its state and covariance within 1e-9 -- no oracle involved."""
    from slam_ros_b200 import EkfFilter
    g = np.load(os.path.join(ROOT, "tests", "golden", "literal_1k.npz"))
    f = EkfFilter(capacity_lines=1000)
    pose = np.zeros(3)

    def step(z, R, enc):
        nonlocal pose
        dX, dY = pose[0] - enc[0], pose[1] - enc[1]
        u = (np.sqrt(dX * dX + dY * dY), 0.0, pose[2] - enc[2])          # Robot.cpp:141-144 (Q5)
        rc, j, pose = f.scan(u, z, R, x_t0=pose)
        assert rc == 0
        return j

    step(g["seed_z"], g["seed_R"], sc.encoder_for(np.zeros(3), np.zeros(3)))
    for s in range(g["u"].shape[0]):
        j = step(g["z"][s], g["R"][s], g["encoder"][s])
        assert (j >= 0).sum() >= 6
        assert np.abs(pose - g["pose"][s]).max() < 1e-9
    L = int(g["L"][0]); nl = 3 + 2 * L
    y, P, Lg = f.download_live()
    pmax = float(g["pmax"][0])
    assert Lg == L and rel(y, g["y"]) < TOL
    assert np.abs(np.diag(P) - g["diag"]).max() / pmax < TOL and np.abs(P[:3] - g["top"]).max() / pmax < TOL
    assert np.abs(P.sum(axis=1) - g["rowsum"]).max() / (pmax * nl) < TOL
    for (r, c), blk in zip(g["corners"], g["blocks"]):
        assert np.abs(P[r:r + blk.shape[0], c:c + blk.shape[1]] - blk).max() / pmax < TOL
