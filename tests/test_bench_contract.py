"""The bench.py contract that can be checked without a GPU: the reference arm (`--impl reference`) prints ONE JSON
line with the keys the driver reads, times a CPU implementation only, and the product arm refuses to run without CUDA."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*argv, timeout=300):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], capture_output=True, text=True, timeout=timeout, cwd=ROOT)


@pytest.mark.parametrize("workload,unit", [("extract", "scans/s"), ("room", "steps/s"), ("10k", "steps/s")])
def test_reference_arm_prints_one_contract_line(workload, unit):
    out = _run("--impl", "reference", "--workload", workload, "--steps", "2", "--warmup", "1")
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, out.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == unit and d["value"] > 0 and d["higher_is_better"] is True
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["gpu_launches"] == 0
    # both arms print the SAME `config` object (the driver compares them): it is built by one function from the workload
    # and the GPU count alone; what a run measured goes to the own arm's `run` object
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.static_config(workload, 1)


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path):
    """--dump-outputs writes the last timed step's results: the same arguments give the same inputs, hence the same
    arrays (what lets two builds be compared output for output), and those arrays are what the CPU oracle computes
    after the same seeded scans."""
    import numpy as np
    from oracle.oracle import StructuredOracle
    from slam_ros_b200 import scenario as sc
    W, K = 3, 4
    dumps = []
    for k in range(2):
        d = tmp_path / ("run%d" % k)
        out = _run("--workload", "1k", "--steps", str(K), "--warmup", str(W), "--no-cpu-baseline", "--dump-outputs", str(d))
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == K
        dumps.append({p.stem: np.load(p) for p in d.glob("*.npy")})
    a, b = dumps
    assert sorted(a) == sorted(b) == ["P_block_origins", "P_blocks", "P_robot_rows", "j", "lines", "pose", "y"]
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for name in a:
        assert a[name].dtype == np.float64 and np.array_equal(a[name], b[name]), name
    L = int(a["lines"][0]); nl = 3 + 2 * L
    j, pose, y, rows, blocks, origins = a["j"], a["pose"], a["y"], a["P_robot_rows"], a["P_blocks"], a["P_block_origins"].astype(int)
    assert j.shape == (8,) and pose.shape == (3,) and y.shape == (nl,) and rows.shape == (3, nl) and blocks.shape == (64, 32, 32)
    assert (j == np.round(j)).all() and (j >= -1).all() and (j < L).all()
    # the pose is y[0:3]; its heading is normalised into (-pi, pi] where y's need not be (a scan without a match)
    assert np.array_equal(y[:2], pose[:2]) and abs(np.angle(np.exp(1j * (y[2] - pose[2])))) < 1e-12
    assert tuple(origins[0]) == (0, 0) and tuple(origins[1]) == (nl - 32, nl - 32)
    for (r0, c0), blk in zip(origins, blocks):
        if r0 == c0:
            assert np.array_equal(blk, blk.T)
        for r in range(r0, min(r0 + 32, 3)):          # rows 0..2 of a block are also in P_robot_rows
            assert np.array_equal(blk[r - r0], rows[r, c0:c0 + 32])
    # the 1k workload, no parity prefix: run_filter draws W + 2K steps of map_scenario(1000, m=8, seed=1) (the timed leg,
    # then the end-to-end leg) for a filter of capacity 1000 + 512; the timed leg ends after step W + K - 1
    scn = sc.map_scenario(1000, W + 2 * K, m=8, seed=1)
    so = StructuredOracle(1512)
    so.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    for s in range(W + K):
        st, jo = so.scan(scn["u"][s], scn["z"][s], scn["R"][s])
    assert L == so.lines and np.array_equal(j, jo)
    assert np.abs(pose - so.pose).max() < 1e-9
    yo, Po = so.live()
    scale = np.abs(Po).max()
    assert np.abs(y - yo).max() / np.abs(yo).max() < 1e-9
    assert np.abs(rows - Po[:3]).max() / scale < 1e-9
    for (r0, c0), blk in zip(origins, blocks):
        assert np.abs(blk - Po[r0:r0 + 32, c0:c0 + 32]).max() / scale < 1e-9


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    out = _run("--steps", "1", "--warmup", "1")
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)
