#!/usr/bin/env python
"""bench.py -- EKF predict+update steps/s at N landmarks, with the covariance sweep's HBM roofline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--dump-outputs DIR]

One "step" = one whole Robot::localize (slam_ros/Robot.cpp:126-943): prediction, association of the m
observed lines against every map landmark, the matched updates (folded into one rank-2m covariance
sweep), augmentation.  Workloads (BASELINE.json `configs`):

    10k      configs[2]  single filter, 10 000 line landmarks (P 20003^2 fp64 = 3.2 GB), m = 8   [default]
    1k       configs[1]  single filter, 1 000 landmarks (P fits L2: launch-bound, not HBM-bound); its CPU baseline /
                         reference arm is the LITERAL reference compiled with LINESIZE = 1000 (oracle/_ref/libslamref1k.so)
    40k      configs[4]  single filter, 40 000 landmarks (51 GB); with --gpus N > 1 row-sharded over N ranks
    mc       configs[3]  Monte-Carlo batch, 4096 independent filters x 50 landmarks, sharded over ranks
    room     configs[0]  the reference-sized filter (LINESIZE=100) on the synthetic room; its CPU baseline /
                         reference arm is the LITERAL reference (oracle/_ref: Robot.cpp compiled over the GSL shim)
    extract  (8f row 2)  line extraction of 361-beam scans (scans/s); CPU baseline = the reference's own
                         lineFitting.cpp (oracle/_ref/libslamlines.so) where built, else the restatement

With --gpus N > 1 (launched by torchrun, one rank per GPU) the default workload runs N independent
filters (replicas; the path needs no collective) -> "scaling": "weak"; `40k` runs ONE filter row-sharded
over the ranks with the per-update NCCL exchange -> "scaling": "strong".

Timing: W warm-up steps, then exactly K steps bracketed by CUDA events recorded on the library's own
stream (ekf_timer_start/stop) after a barrier + synchronize; max over ranks.  The working set (3.2 GB)
is far larger than L2 (126 MB), so no flush is needed between iterations (stated in config.l2).
`value` has the K steps' inputs already resident in HBM (ekf_scan_device); `e2e` drives the public
host-buffer call (ekf_scan: pinned H2D of the step's inputs, D2H of the matches + pose, every step).

The oracle (oracle/) is executed here only as the CPU baseline / reference arm, never as the product.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "10k": dict(N=10000, m=8, headroom=1024, desc="configs[2]: single filter, 10k line landmarks, m=8 batched multi-line updates"),
    "1k": dict(N=1000, m=8, headroom=512, desc="configs[1]: single filter, 1k line landmarks, m=8"),
    "40k": dict(N=40000, m=8, headroom=1024, desc="configs[4]: single filter, 40k line landmarks, m=8"),
    "mc": dict(N=50, m=8, headroom=14, filters=4096, desc="configs[3]: Monte-Carlo batch, 4096 filters x 50 landmarks, m=8"),
    "room": dict(N=100, m=9, headroom=0, desc="configs[0]: the reference-sized filter (LINESIZE=100) on the synthetic 2-D room, 361-beam scans"),
    "extract": dict(N=0, m=0, headroom=0, desc="SURVEY 8f-2: line extraction (mapping_cb + LineExtraction) of 361-beam scans of the synthetic room"),
}


def static_config(wl_name, world, sharded=False, mc_per_gpu=0):
    """The `config` object both arms print (own arm and --impl reference): what is measured, not how it went.
    Run-specific facts (matches per step, exchange path, ...) go to the own arm's `run` object."""
    w = WORKLOADS[wl_name]
    N, m = w["N"], w["m"]
    if wl_name == "mc":
        Bt = mc_per_gpu * world if mc_per_gpu > 0 else w["filters"]
        return {"workload": w["desc"], "landmarks": N, "lines_per_scan": m, "capacity_lines": N + w["headroom"],
                "filters_total": Bt, "parallelism": "independent filters dealt round-robin over %d GPU(s), no collective" % world,
                "l2": "every filter's state is touched once per step; batch state %.0f MB (packed upper triangles) against 126 MB L2; "
                      "no flush between steps" % (Bt * (3 + 2 * N) * (4 + 2 * N) / 2 * 8 / 1e6)}
    if wl_name in ("room", "extract"):
        return {"workload": w["desc"]}
    n = 3 + 2 * N
    par = ("one filter, P row-sharded over %d GPUs" % world) if sharded else ("%d independent filter(s), one per GPU, no collective" % world)
    ws = 8.0 * n * (n + 1) / 2 / 1e9
    l2 = ("per-step working set %.2f GB read + %.2f GB written >> 126 MB L2: no flush needed" % (ws, ws)) if ws > 0.5 else \
         ("P (%.0f MB) fits the 126 MB L2: a latency-bound configuration, no flush between steps (stated, not an HBM-roofline line)" % (ws * 1e3))
    return {"workload": w["desc"], "landmarks": N, "state_dim": n, "lines_per_scan": m, "capacity_lines": N + w["headroom"],
            "parallelism": par, "l2": l2, "seed": "1 (replicas: 1 + rank)"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the structured oracle (port of Robot::localize), all host threads
# ------------------------------------------------------------------------------------------------
def cpu_run(workload, steps, warmup, budget_s, threads=None, n_filters=1, extra_legs=False):
    """Times the CPU restatement of the reference (oracle/ekf_oracle.cpp) on the same workload.  Returns (steps/s, info).

    threads: OpenMP threads of the n^2 row sweeps (None = all host threads; the reference itself has no threads).
    n_filters > 1: the replicas workload at N GPUs -- the host runs the same N independent filters one after the other
    (each with all threads), value = aggregate steps/s over all of them.
    extra_legs: also time ONE step single-threaded (north_star: "reference single-threaded GSL path") and ONE step of
    the -O0 build single-threaded (the reference's CMakeLists sets no optimisation flag), continuing from the same map."""
    from oracle.oracle import StructuredOracle, build
    from slam_ros_b200 import scenario as sc
    build()
    w = WORKLOADS[workload]
    N, m = w["N"], w["m"]
    threads = threads or (os.cpu_count() or 1)
    if workload == "mc":
        # independent filters: one 50-landmark filter is timed on one thread (the natural CPU mapping is a filter per
        # core); batch steps/s = filter-steps/s / filters
        so = StructuredOracle(N + w["headroom"], threads=1)
        scn = sc.map_scenario(N, warmup + steps, m=m, seed=1000)
        so.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
        for s in range(warmup):
            so.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        t0 = time.perf_counter()
        done = 0
        for s in range(warmup, warmup + steps):
            so.scan(scn["u"][s], scn["z"][s], scn["R"][s])
            done += 1
            if time.perf_counter() - t0 > budget_s:
                break
        dt = time.perf_counter() - t0
        fps = done / dt                         # filter-steps per second on one core
        cores = os.cpu_count() or 1
        return fps / w["filters"], {"kind": "port", "cores": 1, "value": fps / w["filters"], "unit": "steps/s", "steps": done,
                                    "all_cores_estimate": {"value": fps * cores / w["filters"], "cores": cores,
                                                           "note": "ESTIMATE: one filter per core, perfect scaling (not measured)"},
                                    "sample": "%d scans of ONE 50-landmark filter on one thread; batch steps/s = filter-steps/s / %d filters (the reference has no threads)" % (done, w["filters"])}
    total_done, total_dt = 0, 0.0
    per_filter_budget = budget_s / max(n_filters, 1)
    legs = {}
    for fi in range(n_filters):
        so = StructuredOracle(N + w["headroom"], threads=threads)
        scn = sc.map_scenario(N, warmup + steps + 2, m=m, seed=1 + fi)
        so.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
        for s in range(min(warmup, 1)):
            so.scan(scn["u"][s], scn["z"][s], scn["R"][s])
        t0 = time.perf_counter()
        done = 0
        for s in range(min(warmup, 1), min(warmup, 1) + steps):
            so.scan(scn["u"][s], scn["z"][s], scn["R"][s])
            done += 1
            if time.perf_counter() - t0 > per_filter_budget:
                break
        total_dt += time.perf_counter() - t0
        total_done += done
        if extra_legs and fi == 0:
            s1 = min(warmup, 1) + done
            so._lib.ekfo_set_threads(so._h, 1)
            t1 = time.perf_counter()
            so.scan(scn["u"][s1], scn["z"][s1], scn["R"][s1])
            legs["single_thread_O2"] = {"value": 1.0 / (time.perf_counter() - t1), "unit": "steps/s", "cores": 1,
                                        "sample": "1 step, g++ -O2, one thread: the reference's own threading (none)"}
            try:
                o0 = StructuredOracle(N + w["headroom"], threads=1, opt0=True)
                o0.adopt(so)
                t1 = time.perf_counter()
                o0.scan(scn["u"][s1 + 1], scn["z"][s1 + 1], scn["R"][s1 + 1])
                legs["single_thread_O0"] = {"value": 1.0 / (time.perf_counter() - t1), "unit": "steps/s", "cores": 1,
                                            "sample": "1 step, g++ -O0 (the reference's CMakeLists.txt:18 sets no optimisation flag), one thread"}
                o0.close()
            except Exception as e:   # noqa: BLE001
                legs["single_thread_O0"] = {"unavailable": str(e)[:120]}
        so.close()
    val = total_done / total_dt
    n = 3 + 2 * N
    # SURVEY section 6: the literal Robot::localize spends 7.1 ms in its dense n^3 prediction dgemms and 0.45 ms per
    # matched line in n^2 passes at n = 203 (LINESIZE = 100, this container's host); scaled, NOT measured
    # + ~0.05 ms per (line, landmark) gate pair; check: the LINESIZE = 1000 build of the reference itself measures 12.7 s
    # per step at n = 2003, m = 8 (bench.py --workload 1k), this formula gives 11.1 s
    lit_ms = 7.1 * (n / 203.0) ** 3 + m * 0.45 * (n / 203.0) ** 2 + m * N * 0.05 * (n / 203.0)
    info = {"kind": "port", "cores": threads, "value": val, "unit": "steps/s", "steps": total_done,
            "literal_reference_extrapolated": "EXTRAPOLATED, not measured: the reference's own dense GSL path would need about "
                                              "%.3g s per step at n = %d (2 n^3 MACs per prediction dgemm)" % (lit_ms / 1e3, n),
            "sample": "%d full steps of the same workload%s on the structured oracle (oracle/ekf_oracle.cpp, the runtime-capacity "
                      "restatement of Robot::localize, bitwise equal to the literal reference where that can run; g++ -O2, OpenMP over "
                      "%d host threads for the n^2 row sweeps; the literal reference is fixed at LINESIZE=100 and cannot run this size)"
                      % (total_done, (" (%d independent filters one after the other, aggregate rate)" % n_filters) if n_filters > 1 else "", threads)}
    info.update(legs)
    return val, info


def _have_literal_1k():
    from oracle.oracle import have_literal_1k
    return have_literal_1k()


def literal_1k_run(steps, budget_s):
    """configs[1] on the reference ITSELF: oracle/_ref/libslamref1k.so = slam_ros/Robot.cpp compiled with
    LINESIZE = 1000 (the two size macros of Robot.h rewritten into a generated header), single thread.  980 landmarks
    (its map resets above LINESIZE - 10); one call is ~12 s (dense n^3 prediction), so the sample is 1-2 steps."""
    from oracle.oracle import LiteralReference
    from slam_ros_b200 import scenario as sc
    N, m = 980, 8
    scn = sc.map_scenario(N, steps + 1, m=m, seed=1)
    lit = LiteralReference(big=True)
    zero = np.zeros(3)
    lit.localize(scn["seed_z"], scn["seed_R"], sc.encoder_for(zero, zero))
    t0 = time.perf_counter(); done = 0
    for s in range(steps):
        y, P, L, pose = lit.state()
        lit.localize(scn["z"][s], scn["R"][s], sc.encoder_for(pose, scn["u"][s]))
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    val = done / dt
    return val, {"kind": "reference", "cores": 1, "value": val, "unit": "steps/s", "steps": done,
                 "sample": "%d Robot::localize calls of the literal reference compiled with LINESIZE=1000 (n = 2003; g++ -O2, GSL shim, "
                           "cout disabled) on a 980-landmark map, m = 8 -- the structured oracle is bitwise equal to it at this size "
                           "(tests/test_oracle.py)" % done}


def room_cpu_run(steps, warmup, budget_s):
    """configs[0] on the host: the reference ITSELF where built (oracle/_ref/libslamref.so = slam_ros/Robot.cpp,
    Q1-patched on a pipe, compiled -O2 over the GSL shim, std::cout disabled (Q14)), else the structured oracle (its
    bitwise restatement, tests/test_oracle.py); single thread either way (the reference has none)."""
    from oracle.oracle import LiteralReference, StructuredOracle, have_literal
    from slam_ros_b200 import scenario as sc
    room = sc.room_scenario(steps=warmup + steps, seed=7, range_sigma=5e-5)
    kind = "reference" if have_literal() else "port"
    if kind == "reference":
        lit = LiteralReference()

        def step(s):
            m = room["count"][s]
            y, P, L, pose = lit.state()
            lit.localize(room["z"][s, :m], room["R"][s, :m], sc.encoder_for(pose, room["u"][s]))
    else:
        so = StructuredOracle(100, threads=1)

        def step(s):
            m = room["count"][s]
            so.localize(room["z"][s, :m], room["R"][s, :m], sc.encoder_for(so.pose, room["u"][s]))
    for s in range(warmup):
        step(s)
    t0 = time.perf_counter()
    done = 0
    for s in range(warmup, warmup + steps):
        step(s)
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    val = done / dt
    what = ("the literal reference (LINESIZE=100, g++ -O2, GSL shim, cout disabled) on the room scenario, including its state "
            "read-back through the harness") if kind == "reference" else \
        "the structured oracle (oracle/ekf_oracle.cpp, capacity 100, g++ -O2, one thread) on the room scenario"
    return val, {"kind": kind, "cores": 1, "value": val, "unit": "steps/s", "steps": done,
                 "sample": "%d Robot::localize calls of %s" % (done, what)}


def run_room(args, rank, world, local):
    """configs[0] on the GPU through the host-buffer call (the drop-in's real use: one small filter, 10 Hz node)."""
    import torch
    from slam_ros_b200 import EkfFilter, scenario as sc
    K, W = args.steps, args.warmup
    torch.cuda.set_device(local)
    room = sc.room_scenario(steps=W + K, seed=7, range_sigma=5e-5)
    f = EkfFilter(capacity_lines=100, device=local)
    f.profile_enable(True)
    for s in range(W):
        m = room["count"][s]
        f.scan(room["u"][s], room["z"][s, :m], room["R"][s, :m])
    f.sync(); f.profile_read()
    clocks = ClockSampler(local); clocks.start()
    t0 = time.perf_counter()
    for s in range(W, W + K):
        m = room["count"][s]
        f.scan(room["u"][s], room["z"][s, :m], room["R"][s, :m])
    f.sync()
    ms = (time.perf_counter() - t0) * 1e3
    clk = clocks.stop()
    prof = f.profile_read()
    peak, peak_src = measured_peaks()
    n = 203
    val = K / (ms / 1e3)
    sweep_ms = prof["sweep_ms"] / max(prof["sweeps"], 1)
    bytes_per_sweep = 8.0 * n * (n + 1)
    return {
        "metric": "EKF predict+update steps/s at N landmarks", "value": val, "unit": "steps/s", "n_gpus": 1, "steps": K, "warmup": W,
        "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOADS["room"]["desc"], "capacity_lines": 100, "lines_per_scan_mean": float(room["count"][W:W + K].mean()),
                   "l2": "P is 330 KB: resident in L2, the path is launch / latency bound (value == e2e: host buffers every step)"},
        "roofline": {"bound": "hbm", "kernel": "k_sweep_pipe", "achieved": bytes_per_sweep / (sweep_ms * 1e-3) / 1e9 if sweep_ms > 0 else 0.0,
                     "peak": peak, "unit": "GB/s", "frac": (bytes_per_sweep / (sweep_ms * 1e-3) / 1e9 / peak) if sweep_ms > 0 else 0.0,
                     "peak_source": peak_src, "launch_ms": sweep_ms, "launches_timed": prof["sweeps"],
                     "algorithmic_bytes_per_launch": bytes_per_sweep, "traffic": None,
                     "note": "not an HBM-bound configuration: 330 KB per sweep"},
        "e2e": {"value": val, "unit": "steps/s", "h2d_bytes_per_step": (6 + 6 * 9) * 8, "d2h_bytes_per_step": 4 * 9 + 128, "ms_per_step": ms / K},
        "gpu_launches": prof["launches"], "clocks": clk,
    }


def lines_cpu_run(steps, budget_s):
    """Line extraction on the host: the reference's own sources (deterministic build) when present, else the port."""
    from oracle.oracle import LinesOracle, LiteralLineExtraction, have_literal_lines
    from slam_ros_b200 import scenario as sc
    kind = "reference" if have_literal_lines() else "port"
    ex = LiteralLineExtraction() if kind == "reference" else LinesOracle()
    S = sc.room_scans(steps=max(steps, 4), seed=17, range_sigma=2e-3)
    ex.extract(S["scans"][0])
    t0 = time.perf_counter(); done = 0
    for s in range(steps):
        ex.extract(S["scans"][s]); done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    what = ("LineExtraction of slam_ros/lineFitting.cpp itself (g++ -O2, GSL shim, zero-initialised locals; it also writes "
            "three text files per call, as in the node)") if kind == "reference" else "oracle/lines_oracle.cpp (g++ -O2)"
    return done / dt, {"kind": kind, "cores": 1, "value": done / dt, "unit": "scans/s", "steps": done,
                       "sample": "%d scans of the same payloads through %s" % (done, what)}


def run_extract(args, rank, world, local):
    """SURVEY 8f row 2: payload -> lines.  value: payloads resident in HBM, results left in HBM (ekf_lx_extract_device,
    K scans enqueued back to back); e2e: host payload in, host lines out, one sync per scan (ekf_lx_extract)."""
    import torch
    from slam_ros_b200 import LineExtractor, scenario as sc
    K, W = args.steps, args.warmup
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    S = sc.room_scans(steps=W + K, seed=17, range_sigma=2e-3)
    scans = S["scans"]; beams = scans.shape[1]
    lx = LineExtractor(device=local)
    d_scans = torch.tensor(scans, dtype=torch.float32, device=dev)
    for s in range(W):
        lx.extract_device(d_scans[s].data_ptr(), beams)
    lx.sync(); torch.cuda.synchronize()
    clocks = ClockSampler(local); clocks.start()
    t0 = time.perf_counter()
    for s in range(W, W + K):
        lx.extract_device(d_scans[s].data_ptr(), beams)
    lx.sync()
    ms = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter(); nl = 0
    for s in range(W, W + K):
        rows, n = lx.extract(scans[s]); nl += n
    e2e_ms = (time.perf_counter() - t0) * 1e3
    clk = clocks.stop()
    peak, peak_src = measured_peaks()
    bytes_per_scan = 8.0 * beams + 6 * 8.0 * beams + 10 * 8.0 * (nl / K)     # payload + point arrays + lines
    return {
        "metric": "line-extraction scans/s (361 beams -> (alfa, r, C_AR, end points) per line)", "value": K / (ms / 1e3), "unit": "scans/s",
        "n_gpus": 1, "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOADS["extract"]["desc"], "beams": int(beams), "lines_per_scan_mean": nl / K,
                   "l2": "a scan is 3 KB: the path is three small dependent kernels, launch / latency bound (no L2 flush applies)"},
        "roofline": {"bound": "hbm", "kernel": "k_lx_segments (one thread block per 0.5 m segment: split recursion + finite-difference covariance)",
                     "achieved": bytes_per_scan / (ms / K * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": bytes_per_scan / (ms / K * 1e-3) / 1e9 / peak, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": bytes_per_scan, "traffic": None,
                     "note": "latency-bound by construction (25 KB per scan); reported for the contract, not a roofline claim"},
        "e2e": {"value": K / (e2e_ms / 1e3), "unit": "scans/s", "h2d_bytes_per_step": int(8 * beams), "d2h_bytes_per_step": 4 + 80 * 128,
                "ms_per_step": e2e_ms / K},
        "gpu_launches": 3 * 2 * K, "clocks": clk,
    }


REF_BUDGET_S = 150.0


def run_reference_arm(args, rank, world):
    """`steps` is the number of steps actually timed: the CPU implementations stop after REF_BUDGET_S seconds of
    timed work, which can be fewer than the --steps requested (`steps_requested`)."""
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    if args.workload == "extract":
        val, info = lines_cpu_run(args.steps, budget_s=REF_BUDGET_S)
        print(json.dumps({"impl": "reference", "metric": "line-extraction scans/s (361 beams -> (alfa, r, C_AR, end points) per line)",
                          "value": val, "unit": "scans/s", "n_gpus": args.gpus, "steps": info["steps"], "steps_requested": args.steps,
                          "budget_s": REF_BUDGET_S, "warmup": args.warmup,
                          "ms_per_step": 1e3 / val, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                          "data": "synthetic", "config": static_config("extract", args.gpus), "cpu_baseline": info,
                          "e2e": {"value": val, "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}), flush=True)
        return
    sharded = args.workload == "40k" and args.gpus > 1
    if args.workload == "1k" and args.lines == 0 and _have_literal_1k():
        val, info = literal_1k_run(args.steps, budget_s=REF_BUDGET_S)
    elif args.workload == "room":
        val, info = room_cpu_run(args.steps, args.warmup, budget_s=REF_BUDGET_S)
    else:
        # replicas at N GPUs = N independent filters: the host runs the same N filters (aggregate rate), so that the
        # driver's ratio compares N GPUs with this one host on the same job
        nf = args.gpus if (args.workload in ("10k", "1k", "40k") and not sharded) else 1
        val, info = cpu_run(args.workload, args.steps, args.warmup, budget_s=REF_BUDGET_S, n_filters=nf)
    line = {
        "impl": "reference", "metric": "EKF predict+update steps/s at N landmarks", "value": val, "unit": "steps/s",
        "n_gpus": args.gpus, "steps": info["steps"], "steps_requested": args.steps, "budget_s": REF_BUDGET_S,
        "warmup": args.warmup, "ms_per_step": 1e3 / val,
        "higher_is_better": True, "scaling": "strong" if (sharded or (args.workload == "mc" and args.mc_per_gpu == 0)) else "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": static_config(args.workload, args.gpus, sharded, args.mc_per_gpu),
        "cpu_baseline": info,
        "e2e": {"value": val, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# own arm
# ------------------------------------------------------------------------------------------------
def _dist_reduce_sum(dev):
    """Sum of per-rank partial read-outs (a row-sharded filter's ranks each emit what they own)."""
    import torch
    import torch.distributed as dist

    def red(a):
        t = torch.tensor(np.ascontiguousarray(a), dtype=torch.float64, device=dev)
        dist.all_reduce(t)
        return t.cpu().numpy()
    return red


DUMP_BLOCKS, DUMP_BLOCK = 64, 32


def dump_filter_outputs(f, j_last, out_dir, rank, red):
    """What a caller of ekf_scan_device holds after the last timed scan, as float64 .npy files in out_dir: that scan's
    association indices (j.npy, -1 = appended), the pose (pose.npy), the landmark count (lines.npy), the live state
    vector (y.npy), the robot rows of the covariance (P_robot_rows.npy, 3 x n) and, since P itself is n^2 doubles
    (3.2 GB at 10k landmarks), DUMP_BLOCKS blocks of DUMP_BLOCK^2 entries of the live covariance: the first and the
    last diagonal block, the others at seeded origins (P_blocks.npy, with their (row, column) origins in
    P_block_origins.npy).  A row-sharded filter's ranks all take part (red sums their partial covariance read-outs;
    y is replicated); rank 0 writes."""
    pose, L, _ = f.state()
    nl = 3 + 2 * L
    y = f.download_y()
    rows = red(f.download_block(0, 0, 3, nl))
    b = min(DUMP_BLOCK, nl)
    origins = np.concatenate([[[0, 0], [nl - b, nl - b]],
                              np.random.default_rng(12345).integers(0, nl - b + 1, size=(DUMP_BLOCKS - 2, 2))])
    blocks = np.stack([red(f.download_block(int(r0), int(c0), b, b)) for r0, c0 in origins])
    if rank != 0:
        return
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("j", j_last), ("pose", pose), ("lines", [L]), ("y", y), ("P_robot_rows", rows), ("P_blocks", blocks),
                    ("P_block_origins", origins)):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def run_filter(wl_name, K, W, rank, world, local, sharded, parity_name=None, exchange_pref="fused", e2e_leg=True, dump_dir=None):
    """One single-filter workload end to end on this rank's GPU (replica, or this rank's shard of a row-sharded filter).
    parity_name: replay the committed oracle fixture tests/golden/oracle_<name>.npz first (same seeded sequence: the
    timing legs then continue from where the fixture ends).  dump_dir: write what the timed leg computed in its last
    step there (dump_filter_outputs).  Returns a dict of raw measurements (rank 0: complete)."""
    import torch
    import torch.distributed as dist
    from slam_ros_b200 import EkfFilter, scenario as sc
    from slam_ros_b200.ekf import nccl_unique_id
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import replay as rp

    w = WORKLOADS[wl_name]
    N, m = w["N"], w["m"]
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    shard = None
    if sharded and world > 1:
        uid = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            uid = torch.tensor(list(nccl_unique_id()), dtype=torch.uint8, device=dev)
        dist.broadcast(uid, 0)
        shard = (rank, world, bytes(uid.cpu().tolist()))
    seed = 1 if (sharded or world == 1) else 1 + rank
    gold = rp.load_golden(parity_name) if parity_name else None
    if gold is not None and (int(gold["N"]) != N or int(gold["m"]) != m or int(gold["cap"]) != N + w["headroom"] or seed != int(gold["seed"])):
        gold = None
    S0 = int(gold["steps"]) if gold is not None else 0
    total_steps = S0 + W + K + (K if e2e_leg else 0)
    scn = sc.map_scenario(N, total_steps, m=m, seed=seed)
    f = EkfFilter(capacity_lines=N + w["headroom"], device=local, shard=shard)
    exchange = None
    if shard is not None:
        # fused exchange over NVLink peer memory inside the line-loop kernel (EKF_SHARD_NCCL=1 keeps the NCCL path)
        from slam_ros_b200.parallel import connect_shards
        fused = exchange_pref == "fused" and os.environ.get("EKF_SHARD_NCCL", "0") != "1" and connect_shards(f, dev)
        exchange = "in-kernel NVLink stores (CUDA IPC peer memory)" if fused else "ncclAllReduce per matched line"
    t_seed = time.perf_counter()
    rc, j, pose = f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    assert rc == 0 and f.lines == N, (rc, f.lines)
    t_seed = time.perf_counter() - t_seed

    parity = None
    if gold is not None:
        sub = {k: (v[:S0] if k in ("u", "z", "R") else v) for k, v in scn.items()}
        r = rp.replay(f, gold, sub, reduce_sum=_dist_reduce_sum(dev) if shard is not None else None)
        parity = {"fixture": "tests/golden/oracle_%s.npz (CPU oracle, made by tests/golden/make_golden_fullsize.py)" % parity_name,
                  "steps": r["steps"], "checkpoints": r["checkpoints"], "assoc_exact": r["assoc_exact"],
                  "first_assoc_mismatch": r["first_assoc_mismatch"], "pose_max_abs_err": r["pose_max_abs_err"],
                  "P_rel_err": r["P_rel_err"], "trace_rel_err": r["trace_rel_err"], "sumsq_rel_err": r["sumsq_rel_err"],
                  "y_rel_err": r["y_rel_err"], "oracle_min_gate_margin": r["oracle_min_gate_margin"],
                  "passed_1e-9": rp.passed(r), "exchange": exchange}
    if K <= 0:
        f.close()
        return {"parity": parity, "exchange": exchange, "seed_s": t_seed}

    # ---- leg 1: inputs resident in HBM --------------------------------------------------------
    lo = S0
    d_u = torch.tensor(scn["u"][lo:], dtype=torch.float64, device=dev)
    d_z = torch.tensor(scn["z"][lo:], dtype=torch.float64, device=dev)
    d_R = torch.tensor(scn["R"][lo:], dtype=torch.float64, device=dev)
    d_j = torch.full((total_steps - lo, m), -7, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()

    def dev_step(s):
        f.scan_device(d_u[s].data_ptr(), m, d_z[s].data_ptr(), d_R[s].data_ptr(), d_j[s].data_ptr())

    for s in range(W):
        dev_step(s)
    f.sync()
    f.profile_read()
    f.profile_enable(True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    f.timer_start()
    for s in range(W, W + K):
        dev_step(s)
    ms = f.timer_stop()
    torch.cuda.synchronize()
    clk = clocks.stop() if rank == 0 else None
    lprof = f.profile_read_lines()
    prof = f.profile_read()
    f.profile_enable(False)
    matched = int((d_j[W:W + K] >= 0).sum().item())
    pose_dev, L_dev, st_dev = f.state()
    if dump_dir:
        dump_filter_outputs(f, d_j[W + K - 1].cpu().numpy(), dump_dir, rank,
                            _dist_reduce_sum(dev) if shard is not None else (lambda a: a))

    # ---- leg 2: end to end through the host-buffer call -------------------------------------------
    e2e_ms, e2e_matched = float("nan"), 0
    if e2e_leg:
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for s in range(lo + W + K, lo + W + 2 * K):
            rc, jj, pose = f.scan(scn["u"][s], scn["z"][s], scn["R"][s])
            e2e_matched += int((jj >= 0).sum())
        f.sync()
        e2e_ms = (time.perf_counter() - t0) * 1e3
    f.close()
    del d_u, d_z, d_R, d_j
    torch.cuda.empty_cache()

    t = torch.tensor([ms, e2e_ms if e2e_leg else 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return {"ms_max": float(t[0]), "e2e_ms_max": float(t[1]) if e2e_leg else None, "ms": ms, "prof": prof, "lprof": lprof, "matched": matched,
            "e2e_matched": e2e_matched, "L": L_dev, "clk": clk, "exchange": exchange, "parity": parity, "seed": seed, "seed_s": t_seed,
            "N": N, "m": m}


def sweep_roofline(r, K, world, sharded):
    """The covariance sweep's roofline entry from the CUDA-event taps of the timed region (rank 0's launches)."""
    n = 3 + 2 * r["L"]
    peak, peak_src = measured_peaks()
    prof, lprof = r["prof"], r["lprof"]
    sweep_ms = prof["sweep_ms"] / max(prof["sweeps"], 1)
    # algorithmic bytes of one sweep: upper triangle read + written once, plus K and KS of the folded
    # terms (SURVEY 8d).  Row-sharded: each rank sweeps 1/world of the triangle (rank 0's share is timed).
    mean_terms = r["matched"] / max(K, 1)
    bytes_per_sweep = (8.0 * n * (n + 1) + 32.0 * n * mean_terms) / (world if sharded else 1)
    achieved = bytes_per_sweep / (sweep_ms * 1e-3) / 1e9 if sweep_ms > 0 else 0.0
    static_traffic = (r["N"] == 10000 and not sharded and r["m"] == 8)
    return {"bound": "hbm", "kernel": "k_sweep_quad (P -= (K S) K' over the upper triangle; TMA + mbarrier ring, 8x4 register tiles, runs under the next scan's line loop)",
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "peak_source": peak_src, "frac_of_nominal_8TBs": achieved / 8000.0,
            "launch_ms": sweep_ms, "launches_timed": prof["sweeps"], "algorithmic_bytes_per_launch": bytes_per_sweep,
            "sweep_share_of_step": (prof["sweep_ms"] / r["ms"]) if r["ms"] > 0 else None,
            "line_stream_ms_per_step": (lprof["line_ms"] / lprof["scans"]) if lprof["scans"] else None,
            "traffic": 3.167e9 if static_traffic else None,
            "traffic_source": ("STATIC, not re-measured by this run (ncu cannot run inside the bench): dram__bytes_read.sum + "
                               "dram__bytes_write.sum per launch from one ncu --set full capture of the same kernel and workload, "
                               "profiles/r1_ncu_sweep_quad.csv (1.615 GB read + 1.552 GB written)") if static_traffic else None}


def run_single_or_replicas(args, rank, world, local, sharded, wl_name=None, parity_name=None):
    import torch
    import torch.distributed as dist
    wl_name = wl_name or args.workload
    w = WORKLOADS[wl_name]
    K, W = args.steps, args.warmup
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
    r = run_filter(wl_name, K, W, rank, world, local, sharded, parity_name=parity_name, dump_dir=args.dump_outputs)
    if rank != 0:
        return None
    filters = 1 if sharded else world
    value = filters * K / (r["ms_max"] / 1e3)
    e2e_value = filters * K / (r["e2e_ms_max"] / 1e3)
    m = w["m"]
    line = {
        "metric": "EKF predict+update steps/s at N landmarks", "value": value, "unit": "steps/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": r["ms_max"] / K, "higher_is_better": True,
        "scaling": "strong" if sharded else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": static_config(wl_name, world, sharded),
        "run": {"matched_per_step": r["matched"] / max(K, 1), "landmarks_at_end": r["L"], "exchange": r["exchange"], "filters": filters,
                "seed_scan_s": r["seed_s"]},
        "roofline": sweep_roofline(r, K, world, sharded),
        "e2e": {"value": e2e_value, "unit": "steps/s", "h2d_bytes_per_step": (6 + 2 * m) * 8 + 4 * m * 8,
                "d2h_bytes_per_step": 4 * m + 128, "ms_per_step": r["e2e_ms_max"] / K, "matched_per_step": r["e2e_matched"] / max(K, 1)},
        "gpu_launches": r["prof"]["launches"],
        "clocks": r["clk"],
    }
    if r["parity"] is not None:
        line["parity"] = r["parity"]
    return line


def run_extras(args, rank, world, local):
    """Driver-visible evidence for the two multi-GPU modes north_star names, attached to the default line as `extra`:
    (i) configs[4], 40k landmarks: ONE filter (row-sharded over the ranks when N > 1, un-sharded at N = 1 so that the
    strong-scaling efficiency can be computed), with the 100-step parity prefix against the committed oracle fixture;
    (ii) configs[3], Monte-Carlo 4096 x 50: the batch split over the ranks (strong) and 4096 filters per GPU (weak);
    (iii) row-sharded parity at 3300 landmarks for BOTH exchange paths (NCCL, fused NVLink) against the oracle fixture."""
    import copy
    import torch
    import torch.distributed as dist
    extra = {}
    K, W = args.steps, args.warmup
    # (i)
    try:
        free_gb = torch.cuda.mem_get_info(local)[0] / 1e9
        need_gb = 2 * 8.0 * 82176.0 ** 2 / 1e9 / world + 4
        if free_gb < need_gb:
            extra["row_sharded_40k"] = {"skipped": "needs %.0f GB of HBM per GPU, %.0f free" % (need_gb, free_gb)}
        else:
            r = run_filter("40k", K, W, rank, world, local, sharded=(world > 1), parity_name="40k")
            if rank == 0:
                rf = sweep_roofline(r, K, world, world > 1)
                extra["row_sharded_40k"] = {
                    "value": K / (r["ms_max"] / 1e3), "unit": "steps/s", "ms_per_step": r["ms_max"] / K, "scaling": "strong",
                    "config": static_config("40k", world, world > 1), "exchange": r["exchange"],
                    "e2e": {"value": K / (r["e2e_ms_max"] / 1e3), "unit": "steps/s", "ms_per_step": r["e2e_ms_max"] / K},
                    "sweep_roofline_per_gpu": {k: rf[k] for k in ("achieved", "peak", "unit", "frac", "launch_ms", "launches_timed",
                                                                   "algorithmic_bytes_per_launch", "sweep_share_of_step")},
                    "line_stream_ms_per_step": rf["line_stream_ms_per_step"],
                    "bound_by": ("sweep" if rf["launch_ms"] >= (rf["line_stream_ms_per_step"] or 0.0) else "line loop"),
                    "matched_per_step": r["matched"] / max(K, 1), "seed_scan_s": r["seed_s"], "parity": r["parity"]}
    except Exception as e:   # noqa: BLE001
        extra["row_sharded_40k"] = {"error": repr(e)[:300]}
    if world > 1:
        dist.barrier()
    # (ii)
    try:
        a = copy.copy(args)
        mc = {}
        a.mc_per_gpu = 0
        ln = run_monte_carlo(a, rank, world, local)
        if rank == 0:
            mc["strong_4096_total"] = {k: ln[k] for k in ("value", "unit", "ms_per_step", "scaling", "e2e")}
            mc["strong_4096_total"].update(filters_per_gpu=ln["run"]["filters_per_gpu"], filter_steps_per_s=ln["run"]["filter_steps_per_s"],
                                           roofline_frac=ln["roofline"]["frac"])
        if world > 1:
            a.mc_per_gpu = 4096
            ln = run_monte_carlo(a, rank, world, local)
            if rank == 0:
                mc["weak_4096_per_gpu"] = {k: ln[k] for k in ("value", "unit", "ms_per_step", "scaling", "e2e")}
                mc["weak_4096_per_gpu"].update(filters_per_gpu=ln["run"]["filters_per_gpu"], filter_steps_per_s=ln["run"]["filter_steps_per_s"],
                                               roofline_frac=ln["roofline"]["frac"])
        extra["mc_4096x50"] = mc
    except Exception as e:   # noqa: BLE001
        extra["mc_4096x50"] = {"error": repr(e)[:300]}
    if world > 1:
        dist.barrier()
    # (iii)
    if world < 2:
        extra["sharded_parity"] = {"skipped": "one process per GPU: needs >= 2 GPUs (the un-sharded replay of the same fixtures is "
                                              "tests/test_gpu_fullsize.py and, for 40k, row_sharded_40k.parity above)"}
    else:
        sp = {}
        WORKLOADS["3300"] = dict(N=3300, m=8, headroom=64, desc="row-sharded parity case, 3300 landmarks (n = 6603: overlapped path)")
        for mode in ("nccl", "fused"):
            try:
                r = run_filter("3300", 0, 0, rank, world, local, sharded=True, parity_name="3300", exchange_pref=mode, e2e_leg=False)
                sp[mode] = r["parity"]
            except Exception as e:   # noqa: BLE001
                sp[mode] = {"error": repr(e)[:300]}
            dist.barrier()
        extra["sharded_parity"] = sp
    return extra if rank == 0 else None


def run_monte_carlo(args, rank, world, local):
    import torch
    import torch.distributed as dist
    from slam_ros_b200 import EkfBatch, scenario as sc

    w = WORKLOADS["mc"]
    N, m, B_total = w["N"], w["m"], w["filters"]
    K, W = args.steps, args.warmup
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
    from slam_ros_b200.parallel import filters_of_rank
    weak = getattr(args, "mc_per_gpu", 0) > 0
    if weak:                                    # weak scaling: a fixed batch per GPU (the 4096-filter batch is the 1-GPU case)
        B_total = args.mc_per_gpu * world
    ids = filters_of_rank(B_total, rank, world)
    B = len(ids)
    cap = N + w["headroom"]
    total = W + 2 * K
    rng_scn = [sc.map_scenario(N, total, m=m, seed=1000 + int(i)) for i in ids[:64]]   # 64 distinct filters, tiled
    reps = (B + len(rng_scn) - 1) // len(rng_scn)
    seed_z = np.concatenate([np.stack([s["seed_z"] for s in rng_scn])] * reps)[:B]
    seed_R = np.concatenate([np.stack([s["seed_R"] for s in rng_scn])] * reps)[:B]
    # step-major host arrays: one step's inputs of the whole batch are contiguous (what a caller hands to ekf_batch_scan)
    U = np.ascontiguousarray(np.concatenate([np.stack([s["u"] for s in rng_scn])] * reps)[:B].transpose(1, 0, 2))          # (total, B, 3)
    Z = np.ascontiguousarray(np.concatenate([np.stack([s["z"] for s in rng_scn])] * reps)[:B].transpose(1, 0, 2, 3))       # (total, B, m, 2)
    Rr = np.ascontiguousarray(np.concatenate([np.stack([s["R"] for s in rng_scn])] * reps)[:B].transpose(1, 0, 2, 3))
    bt = EkfBatch(B, capacity_lines=cap, device=local)
    rc, j, pose = bt.scan(np.zeros((B, 3)), seed_z, seed_R)
    d_u = torch.tensor(U, dtype=torch.float64, device=dev)
    d_z = torch.tensor(Z, dtype=torch.float64, device=dev)
    d_R = torch.tensor(Rr, dtype=torch.float64, device=dev)
    d_j = torch.zeros((B, m), dtype=torch.int32, device=dev)
    for s in range(W):
        bt.scan_device(d_u[s].data_ptr(), m, d_z[s].data_ptr(), d_R[s].data_ptr(), d_j.data_ptr())
    bt.sync()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    for s in range(W, W + K):
        bt.scan_device(d_u[s].data_ptr(), m, d_z[s].data_ptr(), d_R[s].data_ptr(), d_j.data_ptr())
    bt.sync()
    ms = (time.perf_counter() - t0) * 1e3      # the library's stream is its own: host clock around enqueue + sync of K launches
    clk = clocks.stop() if rank == 0 else None
    if world > 1:
        dist.barrier()
    # end to end: every step's inputs come from host memory and its matches + poses go back to host memory; the host
    # path is pipelined two deep (ekf_batch_submit / ekf_batch_collect: the inputs of step s+1 travel under step s's kernel)
    t0 = time.perf_counter()
    bt.submit(U[W + K], Z[W + K], Rr[W + K])
    for s in range(W + K + 1, W + 2 * K):
        bt.submit(U[s], Z[s], Rr[s])
        rc, jj, pose = bt.collect()
    rc, jj, pose = bt.collect()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    bt.close()
    del d_u, d_z, d_R, d_j
    torch.cuda.empty_cache()
    t = torch.tensor([ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank != 0:
        return None
    ms_max, e2e_max = float(t[0]), float(t[1])
    n = 3 + 2 * N                               # live dimension of every filter
    peak, peak_src = measured_peaks()
    bytes_per_launch = 8.0 * n * (n + 1) * B    # upper triangle of every filter read + written once per scan
    achieved = bytes_per_launch / (ms_max / K * 1e-3) / 1e9
    return {
        "metric": "EKF predict+update steps/s at N landmarks", "value": K / (ms_max / 1e3), "unit": "steps/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_max / K, "higher_is_better": True,
        "scaling": "weak" if weak else "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": static_config("mc", world, False, getattr(args, "mc_per_gpu", 0)),
        "run": {"filters_total": B_total, "filters_per_gpu": B, "filter_steps_per_s": B_total * K / (ms_max / 1e3)},
        "roofline": {"bound": "hbm", "kernel": "k_batch_scan (whole localize per CTA; the filter's packed covariance resident in shared memory for the scan: one bulk copy in, one out)",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                     "launch_ms": ms_max / K, "algorithmic_bytes_per_launch": bytes_per_launch, "traffic": None,
                     "note": "not HBM-bound: 8 sequential association gates per filter and scan (fp64 dependency chains) set the time; "
                             "the fraction says how far the batch is from streaming its covariances at HBM speed"},
        "e2e": {"value": K / (e2e_max / 1e3), "unit": "steps/s", "h2d_bytes_per_step": (3 + 6 * m) * 8 * B,
                "d2h_bytes_per_step": (4 * m + 40) * B, "ms_per_step": e2e_max / K},
        "gpu_launches": K, "clocks": clk,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="10k", choices=sorted(WORKLOADS))
    ap.add_argument("--lines", type=int, default=0, help="observed lines per scan (default: the workload's m = 8; "
                    "configs[2] also names m = 32 and 64: one rank-2m sweep per scan)")
    ap.add_argument("--mc-per-gpu", type=int, default=0, help="Monte-Carlo workload: filters PER GPU (weak scaling) instead "
                    "of splitting the 4096-filter batch over the ranks (strong scaling, default)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="default workload only: skip the `extra` object (40k row-sharded / "
                    "un-sharded filter with its parity prefix, Monte-Carlo strong + weak, row-sharded parity on both exchange paths)")
    ap.add_argument("--parity", action="store_true", help="10k / 1k / 40k: replay the committed oracle fixture first and report `parity`")
    ap.add_argument("--cpu-budget", type=float, default=20.0, help="seconds of CPU work for the cpu_baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", help="10k / 1k / 40k: after the timed steps, write what the timed path "
                    "computed in its last step to DIR/<name>.npy (float64; the covariance as a seeded sample of blocks); the "
                    "inputs depend only on the arguments, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload not in ("10k", "1k", "40k")):
        ap.error("--dump-outputs needs the GPU arm (--impl ours) of a single-filter workload (10k, 1k, 40k)")
    if args.lines > 0 and args.workload in ("10k", "1k", "40k"):
        w = WORKLOADS[args.workload]
        w["desc"] = w["desc"].replace("m=%d" % w["m"], "m=%d" % args.lines)
        w["m"] = args.lines
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    rank, world, local = dist_env()
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- libekfcuda has no CPU fallback (use --impl reference for the CPU arm)")
    if args.workload == "mc":
        line = run_monte_carlo(args, rank, world, local)
    elif args.workload == "room":
        line = run_room(args, rank, world, local) if rank == 0 else None
    elif args.workload == "extract":
        line = run_extract(args, rank, world, local) if rank == 0 else None
    else:
        sharded = args.workload == "40k" and world > 1
        line = run_single_or_replicas(args, rank, world, local, sharded,
                                      parity_name=args.workload if (args.parity and args.lines == 0) else None)
        if args.workload == "10k" and args.lines == 0 and not args.no_extras:
            extra = run_extras(args, rank, world, local)
            if rank == 0 and line is not None:
                line["extra"] = extra
    if rank == 0 and line is not None:
        if world == 1 and not args.no_cpu_baseline:
            if args.workload == "extract":
                val, info = lines_cpu_run(steps=200, budget_s=args.cpu_budget)
            elif args.workload == "room":
                val, info = room_cpu_run(steps=1000, warmup=3, budget_s=args.cpu_budget)
            elif args.workload == "1k" and args.lines == 0 and _have_literal_1k():
                val, info = literal_1k_run(steps=2, budget_s=args.cpu_budget)
            else:
                val, info = cpu_run(args.workload, steps=1000, warmup=1, budget_s=min(args.cpu_budget, 6.0), extra_legs=True)
            line["cpu_baseline"] = info
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.barrier()
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
