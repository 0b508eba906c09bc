"""bench.py contract: the reference arm prints ONE JSON line with the agreed keys, and the
helpers that shape the GPU line behave; on a GPU, --dump-outputs writes what the timed steps computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "points/s" and d["higher_is_better"] is True
    assert d["value"] > 1e6 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("interp2_scattered_f64_4096x4096")
    assert d["vs_baseline"] is None and d["dtype"] == "f64" and d["data"] == "synthetic"


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_is_a_seeded_sample_of_the_last_timed_step(tmp_path, oracle):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-extra",
                          "--no-cpu", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout)["steps"] == 2
    files = sorted(os.listdir(tmp_path))
    assert files == ["interp2_scattered_zq.npy"]
    assert sum(os.path.getsize(tmp_path / f) for f in files) <= 64 << 20
    zq = np.load(tmp_path / files[0])
    # the same queries as the timed steps, at the sampled indices, through the CPU oracle: the same bits
    import torch
    import bench
    idx = np.unique(np.random.default_rng(bench.DUMP_SEED).integers(0, bench.NQ, bench.DUMP_SAMPLE))
    assert zq.dtype == np.float64 and zq.shape == idx.shape
    # restates how bench.py main() draws the headline queries on rank 0 (seed 2235 + rank, xq then yq):
    # change both together
    g = torch.Generator(device="cuda").manual_seed(2235)
    xq = torch.rand(bench.NQ, generator=g, device="cuda", dtype=torch.float64)
    yq = torch.rand(bench.NQ, generator=g, device="cuda", dtype=torch.float64)
    some = torch.from_numpy(idx[::50]).cuda()
    ref = oracle.interp2_scattered(*bench.make_grid(), xq[some].cpu().numpy(), yq[some].cpu().numpy())
    assert np.array_equal(zq[::50].view(np.int64), ref.view(np.int64))
