"""bench.py's JSON contract on the CPU-runnable arm (--impl reference), and the static workload maths."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["metric"] == "propagated frames/sec" and d["unit"] == "frames/s"
    assert d["higher_is_better"] is True and d["config"]["workload"] == "davis2017_vos"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == dict(value=d["value"], unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0)
    assert d["value"] > 0 and d["steps"] == 1


def test_reference_arm_dumps_the_last_step(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--dump-outputs", str(tmp_path)], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert sorted(os.listdir(tmp_path)) == ["labels.npy"]
    labels = np.load(tmp_path / "labels.npy")
    assert labels.dtype == np.float32 and labels.shape == (1, 11, 60, 107)
    assert np.abs(labels.sum(axis=1) - 1).max() < 1e-5          # soft labels: weights over the top-k sum to one


def test_dump_outputs_samples_large_arrays_the_same_way_every_time(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    import torch
    masks = torch.randint(0, 11, (64, 480, 854), dtype=torch.uint8, generator=torch.Generator().manual_seed(0))
    small = torch.rand(3, 4, dtype=torch.float64)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), dict(masks=masks, small=small))
    a, b = np.load(tmp_path / "a" / "masks.npy"), np.load(tmp_path / "b" / "masks.npy")
    assert a.dtype == np.float32 and np.array_equal(a, b)
    assert 0 < a.size < masks.numel() and set(np.unique(a)) <= set(range(11))
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), small.numpy())       # float64 kept, not sampled
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 * 1000 * 1000


def test_workload_maths():
    sys.path.insert(0, ROOT)
    import bench
    # SURVEY Appendix B: 60x107, r=12 -> 381.6 in-mask keys per query on average
    pairs = bench.in_mask_pairs(60, 107, 12)
    assert abs(pairs / (60 * 107) - 381.6) < 0.1
    w = bench.algorithmic_work()
    assert w["mem_entries"] == sum(min(t, 20) + 1 for t in range(1, 64))
    assert abs(w["flops_per_step"] - 2 * 256 * pairs * w["mem_entries"]) < 1
    traffic, src = bench.k1_traffic("f16")
    assert traffic is None or traffic > bench.algorithmic_bytes() * 0.5
