"""Cost of one absolute pose fix (ekf_observe_pose) on one GPU, against the same run's 2-term sweep.

Prints JSON lines (and appends them to --out): the card and its power limit; for 10k landmarks (overlapped path) and
40k landmarks, the host-clock time of one full-pose fix (the call plus ekf_sync; the call drains first, so the sweep of
the scans before it is waited for before the clock starts) as min and median over --reps calls, beside
ekf_sweep_probe(m=2) of the same filter; and the steps/s of the 10k, 8-line scan loop with one fix every 10 scans
against none, alternated in one process.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, limit = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": limit}
    except Exception as e:                               # the numbers below are still tied to this run
        return {"gpu": "unknown (%s)" % e, "power_limit": "unknown"}


def seeded(N, cap, steps, seed=11):
    from slam_ros_b200 import EkfFilter, scenario as sc
    scn = sc.map_scenario(N, steps, m=8, seed=seed)
    f = EkfFilter(capacity_lines=cap)
    f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    return f, scn


def fix_args(rng, pose):
    z = np.asarray(pose) + rng.standard_normal(3) * np.array([0.01, 0.01, 0.005])
    R = np.diag([1e-4, 1e-4, 4e-5])
    return z, R


def time_fix(N, cap, reps, rng):
    f, scn = seeded(N, cap, 8)
    for s in range(4):
        f.scan(scn["u"][s], scn["z"][s], scn["R"][s])
    f.observe_pose(*fix_args(rng, f.pose))               # warm-up: first launches of every kernel
    f.sweep_probe(m=2, repeats=3)
    t = []
    for _ in range(reps):
        z, R = fix_args(rng, f.pose)
        f.sync()
        t0 = time.perf_counter()
        f.observe_pose(z, R)
        f.sync()
        t.append((time.perf_counter() - t0) * 1e3)
    probe = [f.sweep_probe(m=2, repeats=10) for _ in range(3)]
    f.close()
    return {"landmarks": N, "fix_ms_min": min(t), "fix_ms_median": float(np.median(t)), "reps": reps,
            "sweep_probe_m2_ms": min(probe), "fix_over_sweep": min(t) / min(probe)}


def steps_per_s(f, scn, s0, steps, every, rng):
    poses = scn["poses"]
    f.sync()
    t0 = time.perf_counter()
    for k in range(steps):
        s = s0 + k
        f.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        if every and k % every == every - 1:
            f.observe_pose(*fix_args(rng, poses[s + 1]))
    f.sync()
    return steps / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--no-40k", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "needs a CUDA device"
    rng = np.random.default_rng(5)

    def emit(r):
        line = json.dumps(r)
        print(line, flush=True)
        if a.out:
            with open(a.out, "a") as fh:
                fh.write(line + "\n")

    emit(dict(card(), what="card"))
    emit(dict(time_fix(10000, 10030, a.reps, rng), what="one fix, 10k (overlapped path)"))
    if not a.no_40k:
        emit(dict(time_fix(40000, 40030, a.reps, rng), what="one fix, 40k, one GPU"))
    f, scn = seeded(10000, 10030, 20 + 2 * a.rounds * a.steps)
    steps_per_s(f, scn, 0, 20, 0, rng)                   # warm-up
    s0, ab = 20, {"none": [], "fix_every_10": []}
    for _ in range(a.rounds):
        for name, every in (("none", 0), ("fix_every_10", 10)):
            ab[name].append(steps_per_s(f, scn, s0, a.steps, every, rng))
            s0 += a.steps
    f.close()
    emit({"what": "10k, 8 lines per scan, steps/s (host loop over ekf_scan), alternated", "rounds": ab,
          "median_none": float(np.median(ab["none"])), "median_fix_every_10": float(np.median(ab["fix_every_10"]))})


if __name__ == "__main__":
    main()
