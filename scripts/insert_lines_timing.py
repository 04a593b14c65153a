"""Time ekf_insert_lines against the same run's device-to-device copy peak and the host round trip it replaces.

    python scripts/insert_lines_timing.py [--reps 5] [--out FILE] [--no-40k]

Cases (DESIGN section 3.3): 100 surveyed walls into 10 000 landmarks; 1 000 landmarks with a full covariance into
10 000; 4 000 landmarks (10 % of the result) into 36 000 on one GPU, surveyed and with a full covariance.  Every
repetition starts from the same map: y and the line count are re-uploaded without P (the insertion writes the same bytes
whatever P holds).  A call ends in a device synchronise, so a host clock around it is the call's time (min and median).
One more call per case runs under torch.profiler, which reports the kernels and the host-to-device copies of the call
separately.  Rates are over the algorithmic bytes written: the new columns of the live upper triangle,
8 (nl_old 2k + 2k (2k + 1) / 2), plus the hot entries (y, rows 0..2 of P, 2x2 diagonal blocks), 8 * 12 k.  The host round
trip (download_live + numpy + upload) is measured once per 10k case.
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


def seeded(N, cap):
    from slam_ros_b200 import EkfFilter, scenario as sc
    scn = sc.map_scenario(N, 2, m=8, seed=3)
    f = EkfFilter(capacity_lines=cap)
    f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    for s in range(2):
        f.scan(scn["u"][s], scn["z"][s], scn["R"][s])
    y = np.zeros(f.n)
    yl = f.download_y()
    y[:yl.size] = yl
    return f, y, f.lines


def spd(k, rng, scale=1e-4):
    A = rng.standard_normal((2 * k, 64))
    M = (A @ A.T / 64 + 0.1 * np.eye(2 * k)) * scale
    return np.triu(M) + np.triu(M, 1).T


def algo_bytes(L, k):
    nl0, w = 3 + 2 * L, 2 * k
    return 8.0 * (nl0 * w + w * (w + 1) / 2), 8.0 * 12 * k


def reset(f, y, L):
    assert f._lib.ekf_upload(f.handle, y.ctypes.data_as(C.POINTER(C.c_double)), None, int(L)) == 0
    f.sync()


def profiled(f, y, L, lines, cov):
    """Device time of one call by kind: the insertion kernels and the host-to-device copies (ms)."""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    reset(f, y, L)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        f.insert_lines(lines, cov)
    out = {"hot_ms": 0.0, "cold_ms": 0.0, "h2d_ms": 0.0, "other_ms": 0.0, "cold_launches": 0}
    for e in prof.events():
        if e.device_type != DeviceType.CUDA:
            continue
        dt, name = e.time_range.elapsed_us() / 1e3, e.name
        if "k_insert_cold" in name:
            out["cold_ms"] += dt; out["cold_launches"] += 1
        elif "k_insert_hot" in name:
            out["hot_ms"] += dt
        elif "HtoD" in name:
            out["h2d_ms"] += dt
        else:
            out["other_ms"] += dt
    return {k: (round(v, 4) if isinstance(v, float) else v) for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--no-40k", action="store_true")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    lines_out = []

    def emit(rec):
        s = json.dumps(rec)
        print(s, flush=True)
        lines_out.append(s)

    name, pl = card()
    peak, tpk = copy_peak()
    emit({"card": name, "power_limit": pl, "copy_peak_GBps": round(peak, 1), "copy_ms_4GB": round(tpk * 1e3, 3)})
    rng = np.random.default_rng(7)
    plan = [(10000, 11100, [("walls100_surveyed", 100, False), ("prior1000_cov", 1000, True)])]
    if not a.no_40k:
        plan.append((36000, 40000, [("tenth4000_surveyed", 4000, False), ("tenth4000_cov", 4000, True)]))
    for N, cap, cases in plan:
        f, y, L = seeded(N, cap)
        for cname, k, with_cov in cases:
            lines = np.stack([rng.uniform(-np.pi, np.pi, k), rng.uniform(2.0, 8.0, k)], axis=1)
            cov = spd(k, rng) if with_cov else None
            ts = []
            for _ in range(a.reps):
                reset(f, y, L)
                t0 = time.perf_counter()
                Ln = f.insert_lines(lines, cov)
                ts.append(time.perf_counter() - t0)
            assert Ln == L + k
            cold, hot = algo_bytes(L, k)
            tmin, tmed = min(ts), float(np.median(ts))
            pr = profiled(f, y, L, lines, cov)
            rec = {"map": L, "case": cname, "inserted": k, "cov": with_cov, "reps": len(ts),
                   "ms_min": round(tmin * 1e3, 3), "ms_median": round(tmed * 1e3, 3),
                   "algo_GB": round((cold + hot) / 1e9, 4), "GBps_call_min": round((cold + hot) / tmin / 1e9, 1),
                   "profiled": pr}
            if pr["cold_ms"] > 0:
                rec["cold_GBps_kernels"] = round(cold / (pr["cold_ms"] / 1e3) / 1e9, 1)
                rec["cold_frac_copy_peak"] = round(cold / (pr["cold_ms"] / 1e3) / 1e9 / peak, 3)
            if with_cov:
                rec["cov_MB"] = round(8.0 * (2 * k) ** 2 / 1e6, 1)
            emit(rec)
            if N == 10000:
                reset(f, y, L)
                t0 = time.perf_counter()
                yl, P, L0 = f.download_live()
                nl0 = yl.size
                Y = np.zeros(f.n); Y[:nl0] = yl; Y[nl0:nl0 + 2 * k] = lines.ravel()
                Pf = np.zeros((f.n, f.n)); Pf[:nl0, :nl0] = P
                del P
                if cov is not None:
                    Pf[nl0:nl0 + 2 * k, nl0:nl0 + 2 * k] = cov
                f.upload(Y, Pf, L0 + k)
                t = time.perf_counter() - t0
                del Pf
                emit({"map": L, "case": cname, "path": "host_round_trip", "ms": round(t * 1e3, 1)})
        f.close()
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as fh:
            fh.write("\n".join(lines_out) + "\n")


if __name__ == "__main__":
    main()
