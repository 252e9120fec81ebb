"""The bench.py output contract, checked on committed records (profiles/r1o_bench_n1.json of round 1, profiles/r2k2_bench_n1.json = the
final line of round 2, both produced on a B200 by `python bench.py`) and on a live `--impl reference` run at a tiny size (CPU only)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config"}


def _check_common(rec: dict):
    assert BASE_KEYS <= set(rec), BASE_KEYS - set(rec)
    baseline = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    # records taken before bench.py read the string from BASELINE.json carry its leading clause only
    assert baseline["metric"].startswith(rec["metric"]) and rec["unit"] == "Mpix/s"
    assert rec["higher_is_better"] is True and rec["vs_baseline"] is None and rec["scaling"] == "weak"
    assert "workload" in rec["config"] and "model" not in rec["config"]
    assert rec["value"] > 0 and rec["ms_per_step"] > 0


@pytest.mark.parametrize("name", ["r1o_bench_n1.json", "r2k2_bench_n1.json"])
def test_committed_gpu_record(name):
    rec = json.loads(open(os.path.join(ROOT, "profiles", name)).read().strip().splitlines()[-1])
    _check_common(rec)
    if name.startswith("r2"):   # round 2: the metric's "PSNR vs ref" half is measured inside the bench, at the benchmarked size
        q = rec["psnr"]
        assert q["size"] == [3840, 2160] and q["frames"] >= 4 and q["pass"] and q["ldr"] >= q["floor_db"] == 49.0
        assert q["reference_storage_vs_fp32_ldr"] < q["ldr"]                       # the kernels sit closer to the fp32 oracle than the reference's render targets do
        assert "r2d_ncu_traffic.json" in rec["roofline"]["traffic_source"] and rec["roofline"]["traffic"] > 0
        assert any("live" in p_ for p_ in rec["passes"]) and rec["config"]["gbuffer"].startswith("renderer formats")
    assert rec["n_gpus"] == 1 and rec["warmup"] >= 3 and rec["dtype"] == "f32" and rec["data"] == "synthetic"
    assert rec["gpu_launches"] >= 20 * rec["steps"]                                  # this library's kernels ran in the timed region
    assert abs(rec["value"] - 3840 * 2160 / 1e6 / (rec["ms_per_step"] / 1e3)) / rec["value"] < 1e-3
    clk = rec["clocks"]
    assert clk["sm_mhz"] and clk["sm_mhz"] > 0.9 * clk["sm_max_mhz"] and not set(clk["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    e2e = rec["e2e"]
    assert e2e["unit"] == rec["unit"] and e2e["h2d_bytes_per_step"] > 0 and e2e["d2h_bytes_per_step"] > 0
    assert e2e["value"] < rec["value"]                                               # host copies are inside its timed region
    roof = rec["roofline"]
    assert roof["bound"] in ("hbm", "tensor") and roof["unit"] == "GB/s" and abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-3
    assert roof["traffic"] is None or roof["traffic"] > 0
    cpu = rec["cpu_baseline"]
    assert cpu["kind"] == "port" and cpu["cores"] >= 1 and cpu["value"] > 0 and cpu["sample"]
    assert abs(sum(p["share"] for p in rec["passes"]) - 1.0) < 0.01
    assert "larger than the 126 MB L2" in rec["config"]["cache"]


def test_reference_arm_live(built):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1", "--ref-width", "160",
                          "--ref-height", "96"], check=True, capture_output=True, text=True, timeout=600).stdout.strip().splitlines()
    assert len(out) == 1, out                                                        # exactly one JSON line
    rec = json.loads(out[0])
    _check_common(rec)
    assert rec["impl"] == "reference" and rec["cpu_baseline"]["value"] == rec["value"]
    # the reference's shaders compiled for the CPU where oracle/_ref exists ("reference"), else the oracle port; the port is always reported beside it
    from oracle.refshader import refsh
    assert rec["cpu_baseline"]["kind"] == ("reference" if refsh.available() else "port") and rec["port"]["value"] > 0
    if rec["cpu_baseline"]["kind"] == "reference":
        assert rec["value"] < rec["port"]["value"] * 1.5          # the checker-grade shader runner is not faster than the port by much, if at all
    assert rec["e2e"] == {"value": rec["value"], "unit": rec["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("dfx_bench", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_dump_outputs_writes_a_fixed_sample_of_the_ldr_plane(tmp_path, monkeypatch):
    import numpy as np
    import torch
    bench = _bench_module()
    ldr = torch.rand((30, 20, 4), generator=torch.Generator().manual_seed(1))
    bench.dump_outputs(str(tmp_path / "whole"), ldr)
    assert np.array_equal(np.load(tmp_path / "whole" / "ldr.npy"), ldr.numpy().reshape(-1, 4))   # small frames: every pixel, raster order
    monkeypatch.setattr(bench, "DUMP_PIXELS", 100)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), ldr)
    a, b = np.load(tmp_path / "a" / "ldr.npy"), np.load(tmp_path / "b" / "ldr.npy")
    assert a.shape == (100, 4) and a.dtype == np.float32 and np.array_equal(a, b)
    flat = ldr.numpy().reshape(-1, 4)
    idx = [int(np.flatnonzero((flat == r).all(axis=1))[0]) for r in a]
    assert idx == sorted(set(idx))                                                    # distinct pixels, ascending raster index


@pytest.mark.gpu
def test_steps_and_dumped_outputs(built, tmp_path):
    """--steps is the number of timed frames (the kernel launches counted in the timed region grow with it in proportion), and
    --dump-outputs writes the last timed frame's LDR plane, the same for the same arguments."""
    import numpy as np

    def run(steps: int, out) -> dict:
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "3", "--width", "320", "--height", "180",
               "--no-cpu-baseline", "--no-psnr", "--dump-outputs", str(out)]
        lines = subprocess.run(cmd, check=True, capture_output=True, text=True, timeout=600).stdout.strip().splitlines()
        assert len(lines) == 1, lines
        return json.loads(lines[0])

    a, b, c = run(2, tmp_path / "a"), run(6, tmp_path / "b"), run(6, tmp_path / "c")
    assert (a["steps"], b["steps"]) == (2, 6) and a["gpu_launches"] >= 40 and b["gpu_launches"] * 2 == a["gpu_launches"] * 6
    ldr = np.load(tmp_path / "b" / "ldr.npy")
    assert ldr.shape == (320 * 180, 4) and ldr.dtype == np.float32 and np.isfinite(ldr).all() and ldr[:, :3].max() > 0
    assert np.array_equal(ldr, np.load(tmp_path / "c" / "ldr.npy"))
