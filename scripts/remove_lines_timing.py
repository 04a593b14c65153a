"""Time ekf_remove_lines against the same run's device-to-device copy peak.

    python scripts/remove_lines_timing.py [--reps 5] [--out FILE] [--no-40k]

Cases (DESIGN section 3.1): 10k landmarks with landmark 0 removed (everything moves), 10 % at random and every other
landmark, each on the out-of-place path (second covariance buffer) and in place (EKF_FLAG_NO_OVERLAP); 40k landmarks on
one GPU with 10 % at random, out of place.  Every repetition starts from the same map: y and the line count are
re-uploaded without P (the compaction moves the same bytes whatever P holds).  A call ends in a device synchronise, so
a host clock around it is the call's time.  Rates are over the algorithmic bytes: read and write of the kept upper
triangle, 8 nl'(nl'+1), plus read and write of the kept hot entries (y, rows 0..2, 2x2 diagonal blocks), 16 (6 nl' - 6).
The host round trip (download_live + np.delete + upload) is measured once at 10k.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # the query is informational; the numbers below do not depend on it
        pl = "unknown (%s)" % e
    return name, pl


def copy_peak(gb=4.0, reps=10):
    """torch device-to-device copy of `gb` GB, CUDA events; GB/s counts read + write."""
    import torch
    n = int(gb * 1e9) // 8
    a = torch.ones(n, dtype=torch.float64, device="cuda"); b = torch.empty_like(a)
    b.copy_(a); torch.cuda.synchronize()
    best = []
    for _ in range(reps):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); b.copy_(a); e1.record(); e1.synchronize()
        best.append(e0.elapsed_time(e1) / 1e3)
    del a, b
    torch.cuda.empty_cache()
    t = min(best)
    return 2 * n * 8 / t / 1e9, t


def seeded(N, flags):
    from slam_ros_b200 import EkfFilter, scenario as sc
    scn = sc.map_scenario(N, 2, m=8, seed=3)
    f = EkfFilter(capacity_lines=N + 64, flags=flags)
    f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    for s in range(2):
        f.scan(scn["u"][s], scn["z"][s], scn["R"][s])
    y = np.zeros(f.n)
    yl = f.download_y()
    y[:yl.size] = yl
    return f, y, f.lines


def algo_bytes(nl):
    return 8.0 * nl * (nl + 1) + 16.0 * (6 * nl - 6)


def time_case(f, y, L, idx, reps):
    lib = f._lib
    ts = []
    for _ in range(reps):
        assert lib.ekf_upload(f.handle, y.ctypes.data_as(C.POINTER(C.c_double)), None, int(L)) == 0
        f.sync()
        t0 = time.perf_counter()
        Ln = f.remove_lines(idx)
        ts.append(time.perf_counter() - t0)
    assert Ln == L - len(idx)
    return ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--no-40k", action="store_true")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    from slam_ros_b200.ekf import EKF_FLAG_NO_OVERLAP
    lines = []

    def emit(rec):
        s = json.dumps(rec)
        print(s, flush=True)
        lines.append(s)

    name, pl = card()
    peak, tpk = copy_peak()
    emit({"card": name, "power_limit": pl, "copy_peak_GBps": round(peak, 1), "copy_ms_4GB": round(tpk * 1e3, 3)})
    rng = np.random.default_rng(7)
    plan = [(10000, "out_of_place", 0), (10000, "in_place", EKF_FLAG_NO_OVERLAP)]
    if not a.no_40k:
        plan.append((40000, "out_of_place", 0))
    for N, path, flags in plan:
        f, y, L = seeded(N, flags)
        sets = {"random10": sorted(rng.choice(L, L // 10, replace=False).tolist())}
        if N == 10000:
            sets = {"landmark0": [0], **sets, "every_other": list(range(0, L, 2))}
        for sname, idx in sets.items():
            ts = time_case(f, y, L, idx, a.reps)
            nl = 3 + 2 * (L - len(idx))
            by = algo_bytes(nl)
            tmin, tmed = min(ts), float(np.median(ts))
            emit({"map": N, "removal": sname, "path": path, "removed": len(idx), "nl_after": nl, "reps": len(ts),
                  "ms_min": round(tmin * 1e3, 3), "ms_median": round(tmed * 1e3, 3), "algo_GB": round(by / 1e9, 3),
                  "GBps_min": round(by / tmin / 1e9, 1), "frac_copy_peak": round(by / tmin / 1e9 / peak, 3)})
        if N == 10000 and path == "out_of_place":
            idx = sets["random10"]
            assert f._lib.ekf_upload(f.handle, y.ctypes.data_as(C.POINTER(C.c_double)), None, int(L)) == 0
            t0 = time.perf_counter()
            yl, P, L0 = f.download_live()
            si = np.array([3 + 2 * j + t for j in idx for t in (0, 1)])
            yl = np.delete(yl, si); P = np.delete(np.delete(P, si, 0), si, 1)
            Y = np.zeros(f.n); Y[:yl.size] = yl
            Pf = np.zeros((f.n, f.n)); Pf[:yl.size, :yl.size] = P
            del P
            f.upload(Y, Pf, L0 - len(idx))
            t = time.perf_counter() - t0
            del Pf
            emit({"map": N, "removal": "random10", "path": "host_round_trip", "ms": round(t * 1e3, 1)})
        f.close()
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
