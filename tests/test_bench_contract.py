"""bench.py prints exactly one JSON line on stdout with the keys the driver reads (both arms)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
             "data", "config", "e2e", "cpu_baseline"}


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, env=e, timeout=900)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def test_reference_arm_line(tmp_path):
    d = _run(["--impl", "reference", "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path)])
    pcm = np.load(tmp_path / "pcm.npy")
    assert pcm.dtype == np.float32 and pcm.shape == (min(os.cpu_count(), 64), 16, 12500)
    assert np.array_equal(pcm, np.rint(pcm)) and np.abs(pcm).sum() > 0
    assert d["impl"] == "reference" and BASE_KEYS <= set(d)
    assert d["unit"] == "Msamples/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "workload" in d["config"]


def test_reference_arm_other_ranks_stay_silent():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, env=dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1"), timeout=300)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_dump_outputs_writes_a_fixed_sample_of_streams(tmp_path):
    import torch

    import bench
    pcm = torch.arange(100 * 16 * 50, dtype=torch.int32).reshape(100, 16, 50).to(torch.int16)
    rssi = np.arange(100 * 16, dtype=np.float32).reshape(100, 16)
    bench.dump_outputs(str(tmp_path / "out"), {"pcm": pcm[:, :, :40], "rssi": rssi})
    pick = np.sort(np.random.default_rng(0).choice(100, bench.DUMP_STREAMS, replace=False))
    got = np.load(tmp_path / "out" / "pcm.npy")
    assert got.dtype == np.float32 and got.shape == (bench.DUMP_STREAMS, 16, 40)
    assert np.array_equal(got, pcm[pick, :, :40].numpy().astype(np.float32))
    assert np.array_equal(np.load(tmp_path / "out" / "rssi.npy"), rssi[pick])
    bench.dump_outputs(str(tmp_path / "all"), {"pcm": pcm[:10]})
    assert np.array_equal(np.load(tmp_path / "all" / "pcm.npy"), pcm[:10].numpy().astype(np.float32))


def test_steps_below_one_are_refused():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert p.returncode == 2 and p.stdout == "" and "--steps" in p.stderr


@pytest.mark.gpu
def test_our_arm_line_small_batch(tmp_path):
    d = _run(["--steps", "2", "--warmup", "1", "--dump-outputs", str(tmp_path)], env={"PMR446_BENCH_STREAMS": "16"})
    pcm = np.load(tmp_path / "pcm.npy")
    assert pcm.dtype == np.float32 and pcm.shape == (16, 16, 12500)
    assert np.array_equal(pcm, np.rint(pcm)) and np.abs(pcm).max() <= 32768 and np.abs(pcm).sum() > 0
    assert BASE_KEYS | {"gpu_launches", "clocks", "roofline", "kernels", "chain_roofline"} <= set(d)
    assert d["n_gpus"] == 1 and d["dtype"] == "f32" and d["vs_baseline"] is None and d["scaling"] == "weak"
    assert d["gpu_launches"] >= 2 * 5 and d["value"] > 0 and d["e2e"]["value"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 16 * 2400000 * 2 and d["e2e"]["d2h_bytes_per_step"] == 16 * 16 * 12500 * 2
    r = d["roofline"]
    assert r["bound"] in ("hbm", "fp32") and {"achieved", "peak", "unit", "frac", "traffic"} <= set(r) and 0 < r["frac"] < 5
    assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"])
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
