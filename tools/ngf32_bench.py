#!/usr/bin/env python
"""GPU: the reference's default configuration -- resnet_6blocks G + 3-layer PatchGAN D, ngf = ndf = 32, BCE
(no_lsgan), 64^3 patches, batch 2 -- on the tensor cores and with every conv forced onto the CUDA-core kernels
(``ops.impl().force_naive``), plus a per-layer table of the six layers whose channel counts are multiples of 32 but not
of 64 (fprop / dgrad / wgrad in ms and TFLOP/s, tensor cores next to CUDA cores).

    python tools/ngf32_bench.py [--steps K] [--warmup W] [--reps R]

The step is timed as bench.py times it: CUDA events around K resident steps replayed as CUDA graphs after W warm-up
steps.  Prints the GPU name and power limit first: the numbers belong to that card."""
import argparse
import contextlib
import io
import os
import random
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mra_gan_b200 import networks3D as N3  # noqa: E402
from mra_gan_b200 import ops  # noqa: E402
from mra_gan_b200.models import create_model  # noqa: E402
from mra_gan_b200.ops import ConvGeom  # noqa: E402
from oracle.ref_import import make_opt  # noqa: E402

PATCH, BATCH = 64, 2
# (name, geometry, input dims): the stem and head see the replication-padded volume (pad 3 on every side)
LAYERS = [
    ("G stem", ConvGeom(1, 32, 7, 1, 0), (PATCH + 6,) * 3),
    ("G.d1", ConvGeom(32, 64, 3, 2, 1), (PATCH,) * 3),
    ("G.u2", ConvGeom(64, 32, 3, 2, 1, True, 1), (PATCH // 2,) * 3),
    ("G head", ConvGeom(32, 1, 7, 1, 0), (PATCH + 6,) * 3),
    ("D.0", ConvGeom(1, 32, 4, 2, 1), (PATCH,) * 3),
    ("D.1", ConvGeom(32, 64, 4, 2, 1), (PATCH // 2,) * 3),
]


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return "nvidia-smi unavailable (%s)" % e


def events_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def step_ms(naive, steps, warmup):
    I = ops.impl()
    I.force_naive = naive
    try:
        random.seed(1234)
        torch.manual_seed(1234)
        opt = make_opt(ngf=32, ndf=32, netG="resnet_6blocks", no_lsgan=True, batch_size=BATCH)
        with contextlib.redirect_stdout(io.StringIO()):
            model = create_model(opt)
            model.setup(opt)
        model.enable_cuda_graphs(warmup_steps=2)
        g = torch.Generator().manual_seed(1234)
        A = (torch.rand((BATCH, 1, PATCH, PATCH, PATCH), generator=g) * 2 - 1).cuda()
        B = (torch.rand((BATCH, 1, PATCH, PATCH, PATCH), generator=g) * 2 - 1).cuda()

        def step():
            model.set_input([A, B])
            model.optimize_parameters()

        for _ in range(max(warmup, 3)):               # two eager steps + the capture step
            step()
        ms = events_ms(step, steps)
        assert I.tc_error() == 0
        losses = model.get_current_losses()
        del model
        return ms, losses
    finally:
        I.force_naive = False


def layer_rows(reps):
    I = ops.impl()
    rows = []
    for name, g, dims in LAYERS:
        gen = torch.Generator().manual_seed(7)
        x = torch.randn((BATCH,) + dims + (g.cin,), generator=gen).to(torch.bfloat16).cuda()
        w = (torch.randn((g.taps, g.cout, g.cin), generator=gen) * 0.02).to(torch.bfloat16).cuda()
        dy = torch.randn((BATCH,) + g.out_dims(dims) + (g.cout,), generator=gen).to(torch.bfloat16).cuda()
        wT = I.pack_weight_t(w, torch.bfloat16)
        od = g.out_dims(dims)
        pos = dims if g.transposed else od
        flop = 2.0 * BATCH * g.cin * g.cout * g.taps * pos[0] * pos[1] * pos[2]
        ops_ = (("fprop", lambda: I.conv_fprop(x, w, None, g)), ("dgrad", lambda: I.conv_dgrad(dy, wT, g, dims)),
                ("wgrad", lambda: I.conv_wgrad(x, dy, g)))
        for op, fn in ops_:
            res = []
            for naive in (False, True):
                I.force_naive = naive
                try:
                    which = ("fprop", "dgrad", "wgrad").index(op)
                    tc = I.conv_uses_tensor_cores(g, BATCH, dims, torch.bfloat16, which)
                    fn(); fn()
                    res.append((events_ms(fn, reps), tc))
                finally:
                    I.force_naive = False
            assert I.tc_error() == 0
            rows.append((name, op, flop, res[0], res[1]))
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20, help="repetitions per layer timing")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "tools/ngf32_bench.py measures on a GPU"
    N3.set_default_compute_dtype(torch.bfloat16)
    print("GPU: %s" % gpu_info())
    print("workload: resnet_6blocks G + 3-layer PatchGAN D, ngf = ndf = 32, BCE, %d^3, batch %d, bf16, CUDA graphs; "
          "%d timed steps after %d warm-up" % (PATCH, BATCH, args.steps, max(args.warmup, 3)))
    ms_tc, l_tc = step_ms(False, args.steps, args.warmup)
    ms_cc, l_cc = step_ms(True, args.steps, args.warmup)
    print("step, tensor-core path                 : %9.2f ms  (%.1f voxels/s)" % (ms_tc, BATCH * PATCH ** 3 / ms_tc * 1e3))
    print("step, every conv on the CUDA cores     : %9.2f ms  (%.1f voxels/s)" % (ms_cc, BATCH * PATCH ** 3 / ms_cc * 1e3))
    print("losses (tensor cores / CUDA cores)     : " + ", ".join("%s %.4f/%.4f" % (k, l_tc[k], l_cc[k]) for k in l_tc))
    print()
    print("%-8s %-6s %9s | %9s %8s %3s | %9s %8s" % ("layer", "op", "GFLOP", "ms", "TFLOP/s", "tc", "ms cuda", "TFLOP/s"))
    for name, op, flop, (t_tc, on_tc), (t_cc, _) in layer_rows(args.reps):
        print("%-8s %-6s %9.2f | %9.4f %8.1f %3s | %9.4f %8.2f" % (name, op, flop / 1e9, t_tc, flop / t_tc / 1e9,
                                                                   "yes" if on_tc else "no", t_cc, flop / t_cc / 1e9))


if __name__ == "__main__":
    main()
