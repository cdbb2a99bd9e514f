"""bench.py --dump-outputs through the command line: two runs with the same arguments write the same arrays bit for bit
(the inputs are seeded and the step adds its partial sums in a fixed order), for the training and the inference workload."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out, *extra):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--no-cpu-baseline",
                        "--no-anchor", "--dump-outputs", str(out)] + list(extra), capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-2000:]
    return sorted(os.listdir(out))


@pytest.mark.parametrize("workload", ["train", "infer"])
def test_dump_outputs_are_reproducible(tmp_path, workload):
    extra = ["--batch", "1"] if workload == "train" else ["--workload", "infer", "--stride", "64"]
    a = _bench(tmp_path / "a", *extra)
    b = _bench(tmp_path / "b", *extra)
    if workload == "train":
        want = ["loss_" + k for k in ("D_A", "G_A", "cycle_A", "idt_A", "D_B", "G_B", "cycle_B", "idt_B")]
        want += ["fake_B", "rec_A", "idt_A", "fake_A", "rec_B", "idt_B", "net_G_A", "net_G_B", "net_D_A", "net_D_B"]
    else:
        want = ["label"]
    assert a == b == sorted(n + ".npy" for n in want)
    for n in a:
        x, y = np.load(str(tmp_path / "a" / n)), np.load(str(tmp_path / "b" / n))
        assert x.dtype in (np.float32, np.float64) and np.isfinite(x).all()
        assert np.array_equal(x, y), n
