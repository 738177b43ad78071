"""bench.py contract checks: the reference arm (CPU oracle port) prints ONE JSON line with the result keys, the
product arm refuses to run without a CUDA device instead of falling back, and on a GPU `--dump-outputs` writes the
last timed step's outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          timeout=timeout, cwd=ROOT)


def test_reference_arm_prints_the_contract_line():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "1", "--shape", "nuscenes")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "lidog_train_scans_per_s" and d["unit"] == "scans/s"
    for key in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["steps"] == 1 and d["warmup"] == 1 and d["higher_is_better"] is True and d["data"] == "synthetic"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == (os.cpu_count() or 1) and cb["value"] == d["value"] and cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the loud failure on a box without a GPU")
def test_product_arm_has_no_cpu_fallback():
    r = _run("--steps", "1", "--warmup", "1", timeout=300)
    assert r.returncode != 0
    assert "CUDA device" in r.stderr and "no CPU fallback" in r.stderr


@pytest.mark.gpu
def test_product_arm_dumps_the_last_timed_step(cuda, tmp_path):
    r = _run("--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(tmp_path), timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["steps"] == 2 and d["warmup"] == 3 and len(d["rank0_step_ms"]) == 2  # two timed steps after three warm-up
    names = sorted(os.listdir(tmp_path))
    assert names == ["buffers.npy", "gradients.npy", "loss.npy", "parameters.npy"]
    assert sum(os.path.getsize(tmp_path / n) for n in names) <= 64 << 20
    for n in names:
        a = np.load(tmp_path / n)
        assert a.dtype in (np.float32, np.float64) and a.size > 0 and np.isfinite(a).all(), n
    assert np.abs(np.load(tmp_path / "gradients.npy")).max() > 0
    # the dumped loss is the 5th training step's (3 warm-up + 2 timed), not that of a later untimed pass:
    # replay bench.py's seeded setup in this process
    from lidog_b200.lidog import bev as lbev, model as M, step, synth
    bench_flag = torch.backends.cudnn.benchmark
    torch.backends.cudnn.benchmark = True
    try:
        torch.manual_seed(1234)
        net = M.MinkUNet34BEV(1, 7, mapping_bound_2d=synth.SHAPES["kitti"]["bound"]).to(cuda)
        if lbev.CONFIG["channels_last"]:
            net.encoders2d.to(memory_format=torch.channels_last)
        trainer = step.LidogTrainer(net, num_classes=7, shape="kitti")
        scans = synth.make_batch(8, 1234, "kitti", 7)
        pts = [torch.from_numpy(p).to(cuda) for p, _ in scans]
        lab = [torch.from_numpy(l).to(cuda) for _, l in scans]
        losses = [float(trainer.training_step(pts, lab)) for _ in range(6)]
    finally:
        torch.backends.cudnn.benchmark = bench_flag
    dumped = float(np.load(tmp_path / "loss.npy"))
    dist = [abs(x - dumped) for x in losses]
    assert dist.index(min(dist)) == 4 and dist[4] <= 1e-4 * abs(dumped), (dumped, losses)
