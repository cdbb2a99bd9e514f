"""bench.py's driver contract on the CPU: the reference arm (`--impl reference`) and the helpers both arms share.

The reference arm is what the driver launches next to the GPU arm (same torchrun command for N > 1): rank 0 alone times
BASELINE config 1 of the oracle port on every host core and prints ONE JSON line; the other ranks exit 0 silently.  The
tests run the arm's own code with the generator / discriminator width cut to 8 filters (a 64-filter 64^3 step takes
~20 s here) -- the line's keys, its `config` object, the thread count and the size fallback do not depend on the width.
"""
import argparse
import io
import json
import os
import subprocess
import sys
from contextlib import redirect_stdout

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

LINE_KEYS = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"}


def _args(**kw):
    d = dict(gpus=1, steps=1, warmup=0, impl="reference", batch=0, no_cpu_baseline=False, no_anchor=False, no_graphs=False,
             workload="train", stride=32, windows_per_pass=4)
    d.update(kw)
    return argparse.Namespace(**d)


@pytest.fixture
def narrow(monkeypatch):
    """cpu_step_seconds with ngf = ndf = 8 (everything else -- sizes asked for, steps, threads -- unchanged)."""
    real = bench.cpu_step_seconds
    calls = []

    def fake(size, steps, warmup, ngf=64):
        calls.append((size, steps, warmup))
        return real(size, steps, warmup, ngf=8)
    monkeypatch.setattr(bench, "cpu_step_seconds", fake)
    return calls


def _run(args, env=None, monkeypatch=None):
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    buf = io.StringIO()
    with redirect_stdout(buf):
        rc = bench.run_reference(args)
    return rc, buf.getvalue()


def test_reference_arm_prints_one_contract_line(narrow, monkeypatch):
    n_before = torch.get_num_threads()
    try:
        monkeypatch.delenv("RANK", raising=False)
        monkeypatch.delenv("WORLD_SIZE", raising=False)
        rc, out = _run(_args(steps=2, warmup=1))
        assert rc == 0
        lines = [l for l in out.splitlines() if l.strip()]
        assert len(lines) == 1
        d = json.loads(lines[0])
        assert set(d) == LINE_KEYS
        assert d["impl"] == "reference" and d["metric"] == "cyclegan_train_voxels_per_sec" and d["unit"] == "voxels/s"
        assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None
        assert d["dtype"] == "f32" and d["data"] == "synthetic" and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1
        # value = voxels of the sample patch / seconds per step; e2e and cpu_baseline repeat the line's own number
        assert d["value"] == pytest.approx(64 ** 3 / (d["ms_per_step"] * 1e-3))
        assert d["e2e"] == {"value": d["value"], "unit": "voxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
        cb = d["cpu_baseline"]
        assert cb["value"] == d["value"] and cb["kind"] == "port" and cb["unit"] == "voxels/s"
        assert "64^3" in cb["sample"] and "BASELINE config 1" in cb["sample"]
        # the config object is the GPU arm's (the driver compares them)
        launch = bench.launch_mode(1)[1]
        assert d["config"] == bench.workload_config(1, bench.default_batch(1), launch)
        assert d["config"]["per_gpu_batch"] == 2 and d["config"]["global_batch"] == 2 and d["config"]["patch"] == 128
        # probe at 32^3, then the timed run at config 1's 64^3 with the steps / warm-up asked for
        assert narrow[0] == (32, 1, 0) and narrow[-1] == (64, 2, 1)
    finally:
        torch.set_num_threads(n_before)


def test_reference_arm_uses_every_host_core_under_torchrun(narrow, monkeypatch):
    """torchrun exports OMP_NUM_THREADS=1 (round 1's reference line was a one-thread run); the arm sets the thread count
    itself and reports it; the N > 1 line carries the N > 1 config (per-GPU batch 4)."""
    n_before = torch.get_num_threads()
    try:
        torch.set_num_threads(1)
        rc, out = _run(_args(gpus=2), env={"RANK": "0", "WORLD_SIZE": "2", "OMP_NUM_THREADS": "1"}, monkeypatch=monkeypatch)
        assert rc == 0
        d = json.loads(out.strip())
        want = len(os.sched_getaffinity(0))
        assert d["cpu_baseline"]["cores"] == want == torch.get_num_threads()
        assert d["n_gpus"] == 2 and d["config"]["parallelism"] == "dp2"
        assert d["config"]["per_gpu_batch"] == 4 and d["config"]["global_batch"] == 8
    finally:
        torch.set_num_threads(n_before)


def test_reference_arm_other_ranks_exit_silently(narrow, monkeypatch):
    rc, out = _run(_args(gpus=8), env={"RANK": "5", "WORLD_SIZE": "8"}, monkeypatch=monkeypatch)
    assert rc == 0 and out == "" and narrow == []


def test_reference_arm_falls_back_to_a_smaller_patch_on_a_slow_host(monkeypatch):
    """The whole --steps K --warmup W run has to end within minutes: a host whose 32^3 probe predicts more than the
    budget for 64^3 gets 48^3 (or 32^3), and the line says so."""
    asked = []

    def fake(size, steps, warmup, ngf=64):
        asked.append(size)
        return {32: 2.0, 48: 6.0, 64: 16.0}[size], 8
    monkeypatch.setattr(bench, "cpu_step_seconds", fake)
    monkeypatch.delenv("RANK", raising=False)
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    rc, out = _run(_args(steps=20, warmup=5))            # 2 s x 8 x 25 = 400 s > 240 s; 2 s x 3.375 x 25 = 169 s fits
    d = json.loads(out.strip())
    assert rc == 0 and asked == [32, 48]
    assert d["value"] == pytest.approx(48 ** 3 / 6.0) and "48^3" in d["cpu_baseline"]["sample"]
    assert "too slow" in d["cpu_baseline"]["sample"]


def test_default_batches_and_launch_modes(monkeypatch):
    monkeypatch.delenv("MRA_DP_GRAPHS", raising=False)
    assert bench.default_batch(1) == 2 and all(bench.default_batch(n) == 4 for n in (2, 4, 8))
    assert bench.launch_mode(1) == (True, "two CUDA graphs per step")
    assert bench.launch_mode(8) == (True, "two CUDA graphs per step")
    assert bench.launch_mode(8, no_graphs=True) == (False, "eager")
    monkeypatch.setenv("MRA_DP_GRAPHS", "0")
    assert bench.launch_mode(1)[0] is True and bench.launch_mode(2)[0] is False
    # model FLOPs per sample-step of SURVEY.md 8(d)
    assert bench.workload_config(1, 2, "eager")["model_tflop_per_sample_step"] == pytest.approx(48.54)


def test_dump_outputs_of_a_training_step(tmp_path, monkeypatch):
    """--dump-outputs: the eight losses (float64), the six generated volumes and the updated weights of the four networks
    (float32) of the model's last step; an output over DUMP_SAMPLE elements as a sample that is the same on every run."""
    import random

    import numpy as np

    from mra_gan_b200 import networks3D as N3
    from mra_gan_b200 import ops
    from mra_gan_b200.models import create_model
    from oracle import functional as OF
    from oracle.ops_ref import RefImpl
    from oracle.ref_import import make_opt
    # a training step dumps 10 tensors: at the full sample size they stay within 64 MB
    assert 10 * bench.DUMP_SAMPLE * 4 <= 64 << 20
    prev = ops.set_impl(RefImpl(torch.float32))
    N3.set_default_compute_dtype(torch.float32)
    try:
        opt = make_opt(ngf=4, ndf=4, pool_size=2, checkpoints_dir=str(tmp_path))
        random.seed(0)
        m = create_model(opt)
        m.setup(opt)
        m.set_input(list(OF.synthetic_patches(1, 32, seed=1)))
        m.optimize_parameters()
        monkeypatch.setattr(bench, "DUMP_SAMPLE", 40000)    # the 32^3 volumes whole, the networks' weights sampled
        for d in ("a", "b"):
            bench.dump_outputs(str(tmp_path / d), bench.step_outputs(m))
        losses = m.get_current_losses()
        vols = ["fake_B", "rec_A", "idt_A", "fake_A", "rec_B", "idt_B"]
        nets = ["G_A", "G_B", "D_A", "D_B"]
        names = ["loss_" + k for k in losses] + vols + ["net_" + n for n in nets]
        assert sorted(os.listdir(tmp_path / "a")) == sorted(n + ".npy" for n in names)
        load = lambda d, n: np.load(str(tmp_path / d / (n + ".npy")))
        for k, v in losses.items():
            a = load("a", "loss_" + k)
            assert a.dtype == np.float64 and a.shape == () and float(a) == v
        for n in vols:
            a = load("a", n)
            assert a.dtype == np.float32 and np.array_equal(a, getattr(m, n).detach().reshape(-1).cpu().numpy())
        for n in nets:
            w = torch.cat([p.detach().reshape(-1) for p in getattr(m, "net" + n).parameters()]).cpu().numpy()
            a = load("a", "net_" + n)
            assert w.size > 40000 and a.dtype == np.float32 and a.shape == (40000,)
            assert np.isin(a, w).all() and np.array_equal(a, load("b", "net_" + n))
    finally:
        ops.set_impl(prev)
        N3.set_default_compute_dtype(torch.bfloat16)


def test_gpu_arm_refuses_to_run_without_a_device():
    """No CPU fallback: without a CUDA device the GPU arm must fail loudly (non-zero exit, no JSON line)."""
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--no-cpu-baseline",
                        "--no-anchor"], capture_output=True, text=True, timeout=300)
    assert p.returncode != 0
    assert not any(l.lstrip().startswith("{") for l in p.stdout.splitlines())
