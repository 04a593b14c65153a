"""A/B of sweep groups (EKF_SWEEP_GROUP, DESIGN section 5) at bench.py's default workload: 10 000 landmarks, m = 8.

In ONE process, filters created with EKF_SWEEP_GROUP=0 (one sweep per scan) and with the default grouping alternate
(the variable is read when a filter is created).  Each run seeds the map, runs --warmup device-resident scans, then times
--steps more with the library's event timer, and prints one JSON line: steps/s, sweep launches per step, sweep ms per
launch, line-stream ms per step, HBM bytes per step of the sweeps (8 n (n + 1) per launch), and the GPU with its power
limit (query-only nvidia-smi).

    python scripts/sweep_group_ab.py [--rounds 3] [--steps 400] [--warmup 50] [--landmarks 10000] [--lines 8]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from slam_ros_b200 import EkfFilter, scenario as sc  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def run(group, N, m, W, K, seed=1):
    if group is None:
        os.environ.pop("EKF_SWEEP_GROUP", None)
    else:
        os.environ["EKF_SWEEP_GROUP"] = str(group)
    scn = sc.map_scenario(N, W + K, m=m, seed=seed)
    f = EkfFilter(capacity_lines=N + 1024)
    rc, _, _ = f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    assert rc == 0 and f.lines == N
    dev = torch.device("cuda")
    d_u = torch.tensor(scn["u"], device=dev); d_z = torch.tensor(scn["z"], device=dev); d_R = torch.tensor(scn["R"], device=dev)
    d_j = torch.full((W + K, m), -7, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()

    def step(s):
        f.scan_device(d_u[s].data_ptr(), m, d_z[s].data_ptr(), d_R[s].data_ptr(), d_j[s].data_ptr())

    for s in range(W):
        step(s)
    f.sync()
    f.profile_read(); f.profile_read_lines()
    f.profile_enable(True)
    f.timer_start()
    for s in range(W, W + K):
        step(s)
    ms = f.timer_stop()
    lines = f.profile_read_lines()
    prof = f.profile_read()
    f.profile_enable(False)
    n = 3 + 2 * f.lines
    matched = int((d_j[W:] >= 0).sum().item())
    f.close()
    return {"EKF_SWEEP_GROUP": "default" if group is None else group, "steps_per_s": K / (ms * 1e-3),
            "ms_per_step": ms / K, "sweep_launches_per_step": prof["sweeps"] / K,
            "sweep_ms_per_launch": prof["sweep_ms"] / max(prof["sweeps"], 1),
            "line_stream_ms_per_step": lines["line_ms"] / max(lines["scans"], 1),
            "hbm_bytes_per_step": 8.0 * n * (n + 1.0) * prof["sweeps"] / K, "matched_per_step": matched / K,
            "landmarks": N, "lines_per_scan": m, "steps": K}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--landmarks", type=int, default=10000)
    ap.add_argument("--lines", type=int, default=8)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("sweep_group_ab.py needs a CUDA device")
    gpu = gpu_info()
    for _ in range(a.rounds):
        for group in (0, None):
            r = run(group, a.landmarks, a.lines, a.warmup, a.steps)
            r["gpu"] = gpu
            print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
