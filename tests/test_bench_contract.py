"""bench.py contract on CPU: the reference arm runs the unmodified reference decoder (oracle/_ref) or the oracle port on
the host cores and prints one JSON line with the agreed keys."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--sample-iters", "1"], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads(p.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["unit"] == "edge-updates/s" and d["higher_is_better"] is True
    assert d["value"] > 1e6 and d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert "L=50 M=10000" in d["config"]["workload"]


def test_dump_outputs_writes_every_result_and_samples_above_the_limit(tmp_path, monkeypatch):
    import numpy as np
    import torch
    import bench
    res = torch.arange(5 * 2 * 300, dtype=torch.int32).reshape(5, 2, 300)
    bench.dump_outputs(str(tmp_path / "all"), res)
    for i, name in enumerate(bench.DUMP_NAMES):
        a = np.load(tmp_path / "all" / (name + ".npy"))
        assert a.dtype == np.float64 and (a == res[i].numpy()).all()
    assert not (tmp_path / "all" / "frame_ids.npy").exists()
    monkeypatch.setattr(bench, "DUMP_LIMIT", 8 * 11 * 100)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), res)
    ids = np.load(tmp_path / "s1" / "frame_ids.npy").astype(np.int64)
    assert len(ids) == 100 and (np.diff(ids) > 0).all() and (ids == np.load(tmp_path / "s2" / "frame_ids.npy")).all()
    total = sum(os.path.getsize(tmp_path / "s1" / f) for f in os.listdir(tmp_path / "s1"))
    assert total < 8 * 11 * 100 + 6 * 256                     # data within the limit, plus the .npy headers
    for i, name in enumerate(bench.DUMP_NAMES):
        assert (np.load(tmp_path / "s1" / (name + ".npy")) == res[i].numpy()[:, ids]).all()


def test_non_zero_ranks_of_the_reference_arm_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""
