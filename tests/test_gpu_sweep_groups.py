"""Sweep groups: consecutive overlapped scans share one covariance sweep (EKF_SWEEP_GROUP, DESIGN section 5).

Every case runs twice in a child process, once with one sweep per scan (EKF_SWEEP_GROUP=0, the reference) and once with
the default grouping, and the two runs must agree bit for bit: per-scan matches and pose, y, cov_stats and covariance
blocks that include the newest columns.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CHILD = r'''
import sys, numpy as np, torch
sys.path.insert(0, ROOT)
from slam_ros_b200 import EkfFilter, scenario as sc
out = {}

def blocks(f, key, extra=()):
    y = f.download_y()
    n = len(y)
    out["y_" + key] = y
    out["S_" + key] = np.array(f.cov_stats())
    t = max(n - 64, 0)
    spots = [(0, 0), (3, 3), (5, 900), (t, t), (0, t), (max(n - 200, 0), t)] + list(extra)
    out["B_" + key] = np.stack([f.download_block(r0, c0, 64, 64) for r0, c0 in spots])

def seeded(N, cap, scn):
    f = EkfFilter(capacity_lines=cap)
    f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    return f

def ghost_z(world_line, pose):
    return sc.observe(np.asarray(world_line, dtype=np.float64)[None, :], pose)[0]

# 1. m = 8: a line that is new in the first scan of a group and matched, as that new landmark, in the second
#    (register-resident line loop at 3 300 landmarks, memory-resident at 12 000)
for N in (3300, 12000):
    steps = 8
    scn = sc.map_scenario(N, steps, m=8, seed=11)
    f = seeded(N, N + 96, scn)
    J, X = [], []
    for s in range(steps):
        z = scn["z"][s].copy()
        g = scn["world"][(5 * s) % N].copy(); g[1] += 3.0            # a ghost of a true line: matches nothing in the map
        if s % 2 == 0:
            ghost = g
            z[1] = ghost_z(ghost, scn["poses"][s + 1])
        else:
            z[1] = ghost_z(ghost, scn["poses"][s + 1])               # the previous scan's ghost, now a landmark
        rc, j, pose = f.scan(scn["u"][s], z, scn["R"][s])
        J.append(j); X.append(pose)
    key = "ghost_%d" % N
    out["J_" + key] = np.stack(J); out["X_" + key] = np.stack(X)
    blocks(f, key)
    f.close()

# 2. line counts that close groups for every reason: budget, line-loop class (m > 8 takes more SMs at this capacity),
#    chunked scan (40 lines), empty scan
N = 12000
ms = [8, 3, 5, 12, 1, 16, 0, 8, 40, 5, 3, 8, 12, 12, 1, 1, 1, 8]
scn = sc.map_scenario(N, len(ms), m=40, seed=13)
f = seeded(N, N + 96, scn)
J, X = [], []
for s, m in enumerate(ms):
    z = scn["z"][s, :m].copy()
    if m >= 3: z[2, 1] += 3.0
    rc, j, pose = f.scan(scn["u"][s], z, scn["R"][s, :m])
    J.append(np.pad(j, (0, 40 - m), constant_values=-7)); X.append(pose)
out["J_mixed"] = np.stack(J); out["X_mixed"] = np.stack(X)
blocks(f, "mixed")
f.close()

# 3. a map reset as the first scan of a group, on the overlapped path (device-resident scans: the host only has an
#    upper bound of the map size, so the scans after the reset stay on the pipeline); the rebuilt map re-observes half
#    of the previous scan's lines, so later scans match landmarks appended in the scan before
N, steps = 3300, 16
scn = sc.map_scenario(N, steps, m=8, seed=17, stride=4)
f = EkfFilter(capacity_lines=N + 45)                      # 4 growing scans fit (+32), the fifth (+40) resets
f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
z = scn["z"].copy()
for s in range(5): z[s, :, 1] += 3.0 + 0.5 * s             # lines that match nothing: the map grows by 8 per scan
dev = torch.device("cuda")
d_u = torch.tensor(scn["u"], device=dev); d_z = torch.tensor(z, device=dev); d_R = torch.tensor(scn["R"], device=dev)
d_j = torch.zeros((steps, 8), dtype=torch.int32, device=dev)
for s in range(steps):
    f.scan_device(d_u[s].data_ptr(), 8, d_z[s].data_ptr(), d_R[s].data_ptr(), d_j[s].data_ptr())
f.sync()
pose, L, _ = f.state()
out["J_reset"] = d_j.cpu().numpy(); out["X_reset"] = pose; out["L_reset"] = np.array([L])
assert L < 200, L                                          # the reset happened
blocks(f, "reset", extra=((3, max(3 + 2 * L - 64, 0)),))
f.close()

# 4. every observer of the covariance with a group open: download_block, sweep_probe, a step-wise scan, sync; and the
#    timer around an odd number of scans accounts for the sweep of every term those scans produced
N = 3300
scn = sc.map_scenario(N, 12, m=8, seed=19)
f = seeded(N, N + 96, scn)
B = []
def scan(s):
    return f.scan(scn["u"][s], scn["z"][s], scn["R"][s])[1]
J = [scan(0)]
B.append(f.download_block(0, 0, 64, 64)); B.append(f.download_block(3, 2 * N - 61, 64, 64))
J.append(scan(1)); J.append(scan(2)); J.append(scan(3))
f.sweep_probe(m=3, repeats=1)
B.append(f.download_block(3, 2 * N - 61, 64, 64))
J.append(scan(4))
f.predict(scn["u"][5])
for i in range(8):
    zi, Ri = scn["z"][5, i], scn["R"][5, i]
    j, _ = f.associate(zi, Ri)
    if j >= 0: f.update(j, zi, Ri)
    else: f.add_line(zi, Ri)
f.end_scan(8)
J.append(scan(6))
f.sync()
B.append(f.download_block(3, 2 * N - 61, 64, 64))
J.append(scan(7))
f.sync()
f.profile_read(); f.profile_enable(True)
f.timer_start()
for s in (8, 9, 10):
    J.append(scan(s))
f.timer_stop()
prof = f.profile_read()
f.profile_enable(False)
n = 3.0 + 2.0 * f.lines
terms = (prof["sweep_bytes"] - prof["sweeps"] * 8.0 * n * (n + 1.0)) / (32.0 * n)
assert round(terms) == 24, (prof, terms)                   # every one of the three scans' 8 terms was swept
out["J_flush"] = np.stack(J); out["B_flush"] = np.stack(B)
blocks(f, "flush")
f.close()
np.savez(sys.argv[1], **out)
'''.replace("ROOT", repr(ROOT))


def _run(group):
    path = "/tmp/ekf_sweep_group_%s_%d.npz" % (group or "default", os.getpid())
    env = dict(os.environ)
    env.pop("EKF_SWEEP_GROUP", None)
    if group is not None:
        env["EKF_SWEEP_GROUP"] = group
    out = subprocess.run([sys.executable, "-c", CHILD, path], capture_output=True, text=True, timeout=1200, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    res = dict(np.load(path))
    os.remove(path)
    return res


def test_sweep_groups_give_identical_bits(libekf):
    ref = _run("0")
    grp = _run(None)
    assert set(ref) == set(grp)
    for k in sorted(ref):
        assert np.array_equal(ref[k], grp[k]), k
    # the cases exercise what they are meant to: ghosts matched in the next scan, new landmarks after the reset
    for N in (3300, 12000):
        J = ref["J_ghost_%d" % N]
        assert (J[0::2, 1] < 0).sum() >= 2 and (J[1::2, 1] >= N).sum() >= 2, J[:, 1]
    assert (ref["J_reset"][6:] >= 0).sum() > 10
