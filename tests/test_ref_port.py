"""The CPU baseline port (oracle/ref_port.py, what bench.py times as the reference arm) must
compute what the reference computes: checked against the golden vectors of the real reference."""
import numpy as np
import torch

import cmax_scenes
from conftest import assert_close_to_max, golden
from oracle import ref_port


def test_voxel_ports():
    g = golden("voxel_torch")
    for tag in "abd":
        out = ref_port.voxel_torch_cpu(*(torch.from_numpy(g[tag + k]) for k in ("_x", "_y", "_t", "_p")),
                                       int(g[tag + "_B"]), tuple(int(v) for v in g[tag + "_HW"]))
        assert_close_to_max(out.numpy(), g[tag + "_out"], 1e-6, tag)
    g = golden("voxel_numpy")
    for tag in "ab":
        out = ref_port.voxel_numpy(g[tag + "_x"], g[tag + "_y"], g[tag + "_t"], g[tag + "_p"], int(g[tag + "_B"]),
                                   tuple(int(v) for v in g[tag + "_HW"]))
        assert_close_to_max(out, g[tag + "_out"], 1e-12, tag)


def test_cmax_port():
    g = golden("cmax")
    for row in g["evals"][::5]:
        s, vx, vy, sigma, f_ref, g0, g1 = row
        tag = {0: "c9", 1: "lat"}[int(s)]
        f, gr = ref_port.cmax_fg_cpu((vx, vy), *cmax_scenes.events(g, tag), (180, 240), sigma)
        assert abs(f - f_ref) <= 1e-6 * abs(f_ref) + 1e-12
        assert np.abs(gr - np.array([g0, g1])).max() <= 1e-5 * max(abs(g0), abs(g1)) + 1e-9


def test_reference_arm_prints_the_contract_line(tmp_path):
    """`bench.py --impl reference` (the arm the driver runs beside ours): one JSON line on stdout with the
    contract's keys, on a reduced sample so that the test stays short; needs no GPU."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, EVK_BENCH_CPU_SAMPLE="200000", EVK_BENCH_EVENTS="1000000", EVK_BENCH_REF_BUDGET_S="10")
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, env=env, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "Mevents/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert 1 <= line["config"]["reference_events_per_step"] <= 1_000_000
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["value"] == line["value"]
    grid = np.load(tmp_path / "voxel.npy")           # --dump-outputs: the grid of the last timed step
    assert grid.shape == (5, 480, 640) and grid.dtype == np.float32 and np.isfinite(grid).all() and grid.any()
