#!/usr/bin/env python
"""Benchmark of the CycleGAN training hot path (BASELINE.json metric: train voxels/sec at 128^3).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this framework on N B200s
    python bench.py --impl reference [...]                         # the reference's CPU path (oracle port)
    python bench.py [...] --dump-outputs DIR                       # + what the last timed step computed, as DIR/*.npy

N > 1 is launched by torchrun (one rank per GPU, NCCL).  A "step" is one
``CycleGANModel.optimize_parameters()`` on a synthetic U(-1,1) 128^3 batch; rank 0 prints ONE JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PATCH = 128
FLOP_PER_SAMPLE_STEP = 48.540e12        # SURVEY.md 8(d): conv MACs x2, fwd+dgrad+wgrad, 128^3


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p, "measured"
    except Exception:  # noqa: BLE001
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:  # noqa: BLE001
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for nm, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        # samples taken while the GPU was busy = upper half of the distribution
        busy = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": busy[len(busy) // 2] if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_opt(**kw):
    ns = argparse.Namespace(
        gpu_ids=0, isTrain=True, checkpoints_dir="/tmp/mra_bench_ckpt", name="bench", input_nc=1, output_nc=1,
        ngf=64, ndf=64, netG="resnet_9blocks", netD="n_layers", n_layers_D=3, norm="instance", no_dropout=True,
        init_type="normal", init_gain=0.02, no_lsgan=False, pool_size=50, lr=2e-4, beta1=0.5, lambda_A=10.0,
        lambda_B=10.0, lambda_identity=0.5, lambda_co_A=2, lambda_co_B=2, which_direction="AtoB",
        lr_policy="lambda", epoch_count=1, niter=500, niter_decay=100, lr_decay_iters=50, continue_train=False,
        which_epoch="latest", verbose=False, model="cycle_gan", model_suffix="", batch_size=1)
    for k, v in kw.items():
        setattr(ns, k, v)
    return ns


WORKLOAD = ("resnet_9blocks G + 3-layer PatchGAN D, ngf=ndf=64, LSGAN, one CycleGAN optimize_parameters() on "
            "synthetic 128^3 patches")
# --workload unet = BASELINE config 4 (the 7-down UNet as both generators), --workload infer = config 5 (sliding window)
WORKLOAD_UNET = ("unet_128 (7-down UNet) G + 3-layer PatchGAN D, ngf=ndf=64, LSGAN, one CycleGAN optimize_parameters() "
                 "on synthetic 128^3 patches (BASELINE config 4)")
WORKLOAD_INFER = ("sliding-window G_A inference (test.py path): resnet_9blocks ngf=64 over a synthetic 256x256x160 volume, "
                  "128^3 windows, stride %d/%d = %d windows sharded over the ranks, one reduce to rank 0 (BASELINE config 5)")
FLOP_PER_SAMPLE_STEP_UNET = 5.245e12    # SURVEY.md 8(d)
G_FWD_FLOP_PER_WINDOW = 2.619e12        # resnet_9blocks forward on one 128^3 window (SURVEY.md 8a: 1309.7 GMAC)


def default_batch(world):
    """BASELINE.json: config 2 (1 GPU) is quoted at batch 2, config 3 (2/4/8 GPUs) at batch 4 per GPU."""
    return 2 if world == 1 else 4


def workload_config(world, per_gpu_batch, launch, workload="train"):
    """The `config` object of the JSON line -- the SAME for this framework's arm and for --impl reference (whose steps
    are a bounded CPU sample of this workload, described in its cpu_baseline.sample)."""
    unet = workload == "unet"
    return {"workload": WORKLOAD_UNET if unet else WORKLOAD, "patch": PATCH, "per_gpu_batch": per_gpu_batch,
            "global_batch": per_gpu_batch * world, "parallelism": "dp%d" % world,
            "l2": "per-step working set (tens of GB) >> 126 MB L2", "launch": launch,
            "model_tflop_per_sample_step": (FLOP_PER_SAMPLE_STEP_UNET if unet else FLOP_PER_SAMPLE_STEP) / 1e12}


def launch_mode(world, no_graphs=False):
    use_graphs = not no_graphs and (world == 1 or os.environ.get("MRA_DP_GRAPHS", "1") == "1")
    return use_graphs, ("two CUDA graphs per step" if use_graphs else "eager")


# ------------------------------------------------------------------------------------------------
# CPU baseline: the reference's algorithm (oracle port) on the host cores
# ------------------------------------------------------------------------------------------------
def use_all_host_cores():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core (and says how many)."""
    import torch
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0)) or n
    except Exception:  # noqa: BLE001
        pass
    torch.set_num_threads(n)
    return torch.get_num_threads()


def cpu_step_seconds(size, steps, warmup, ngf=64):
    import random

    import torch

    from oracle import functional as OF
    use_all_host_cores()
    random.seed(1234)
    sds = OF.build_cyclegan_weights(ngf, ngf, seed=1234)
    m = OF.CycleGANOracle(*sds, netG="resnet_9blocks", no_lsgan=False)
    times = []
    for s in range(warmup + steps):
        A, B = OF.synthetic_patches(1, size, seed=1234 + s)
        t0 = time.perf_counter()
        m.optimize_parameters(A, B)
        float(m.losses["G"].detach())
        if s >= warmup:
            times.append(time.perf_counter() - t0)
    return sum(times) / len(times), torch.get_num_threads()


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port; the reference is pure Python
    on torch CPU with no setup.py, so there is nothing to pip-install or compile), on all host cores.  Each step is
    BASELINE config 1 -- one optimize_parameters() on a 64^3 patch, batch 1, fp32 -- a bounded sample of the 128^3
    workload (voxels/s is size-normalised); a slower host falls back to 48^3 / 32^3 to keep the run within minutes."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return 0
    import torch
    threads = use_all_host_cores()
    t_small, _ = cpu_step_seconds(32, 1, 0)
    budget = 240.0
    size = 32
    for cand in (64, 48):
        if t_small * (cand / 32.0) ** 3 * (args.steps + args.warmup) < budget:
            size = cand
            break
    sec, threads = cpu_step_seconds(size, args.steps, args.warmup)
    vox = size ** 3 / sec
    _, launch = launch_mode(world)
    sample = ("each step = one optimize_parameters() of the oracle port on a %d^3 patch, batch 1, fp32%s; %d timed "
              "step(s) after %d warm-up, %d host threads, torch CPU %s"
              % (size, " (BASELINE config 1)" if size == 64 else " (host too slow for config 1's 64^3 within the time budget)",
                 args.steps, args.warmup, threads, torch.__version__))
    line = {
        "impl": "reference", "metric": "cyclegan_train_voxels_per_sec", "value": vox, "unit": "voxels/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(world, args.batch if args.batch else default_batch(world), launch),
        "cpu_baseline": {"value": vox, "unit": "voxels/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": vox, "unit": "voxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def cpu_baseline_block():
    """Bounded CPU sample for the GPU arm's line: BASELINE config 1 (64^3, batch 1, fp32), 2nd and 3rd step."""
    sec, threads = cpu_step_seconds(64, 2, 1)
    return {"value": 64 ** 3 / sec, "unit": "voxels/s", "cores": threads, "kind": "port",
            "sample": "BASELINE config 1: 64^3 patch, batch 1, fp32; mean of steps 2-3 of optimize_parameters() "
                      "(%.1f s each) of the oracle port on %d host threads" % (sec, threads)}


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def time_dominant_kernel(torch, I, batch, reps=20):
    """The dominant kernel: the 256->256 k3 conv on the padded 34^3 tensor (G.rb fprop = gather_halo_kernel,
    79.7 % of generator FLOPs).  Timed alone with CUDA events on the launching stream."""
    from mra_gan_b200.ops import ConvGeom
    g = ConvGeom(256, 256, 3, 1, 0)
    x = torch.randn((batch, 34, 34, 34, 256), device="cuda").to(torch.bfloat16)
    w = (torch.randn((27, 256, 256), device="cuda") * 0.02).to(torch.bfloat16)
    flush = torch.empty(192 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    for _ in range(3):
        I.conv_fprop(x, w, None, g, want_stats=True)
    total = 0.0
    for _ in range(reps):
        flush.zero_()                                  # evict the operands from L2 between launches
        torch.cuda._sleep(600000)                      # ~0.3 ms spin kernel: the host queues the launch behind it, so the
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)   # events bracket device time
        e0.record()                                    # only (no Python / ctypes / tensor-map-encode latency inside)
        I.conv_fprop(x, w, None, g, want_stats=True)
        e1.record()
        e1.synchronize()
        total += e0.elapsed_time(e1)
    ms = total / reps
    flops = 2.0 * batch * 32 ** 3 * 256 * 256 * 27
    return ms, flops


def time_norm_kernels(torch, I, batch, hbm_peak, reps=10):
    """HBM-bound companions of the conv kernel: the fused InstanceNorm+ReLU(+pad) forward and backward on the
    largest activation of the generator (64 channels x 128^3, G.c1 / G.u2 norms).  Algorithmic bytes
    (SURVEY.md 8d): fwd = read x + write y, bwd = read gy + read x + write dx; the tensors (0.5 GB each at batch 2)
    are far larger than L2, so no flush is needed between launches."""
    from mra_gan_b200.ops import ACT_RELU
    x = torch.randn((batch, 128, 128, 128, 64), device="cuda").to(torch.bfloat16)
    stats = I.inorm_stats(x)
    y, mean, rstd = I.inorm_fwd(x, stats, None, 0, ACT_RELU, 0.0, -1)
    gy = torch.randn_like(y)
    e = x.numel() * 2

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        torch.cuda._sleep(3000000)                     # ~1.5 ms spin kernel: lets the host run ahead of the device
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / reps

    sums = I.inorm_bwd_stats(gy, x, mean, rstd, 0, ACT_RELU, 0.0, -1)
    t_f = timed(lambda: I.inorm_fwd(x, stats, None, 0, ACT_RELU, 0.0, -1))
    t_a = timed(lambda: I.inorm_bwd_apply(gy, x, mean, rstd, sums, 0, ACT_RELU, 0.0, -1))
    t_b = timed(lambda: I.inorm_bwd(gy, x, mean, rstd, 0, ACT_RELU, 0.0, -1))
    out = []
    for name, ms, nbytes, launches in (
            ("inorm_fwd_stream_kernel (IN+ReLU fwd, 64ch x 128^3)", t_f, 2 * e, 1),
            ("inorm_bwd_stream_kernel (IN+ReLU bwd, 64ch x 128^3: what the step runs on this tensor -- the reduction "
             "pass {sum dy, sum dy xhat} comes out of the consumer conv's dgrad epilogue, mra_conv3d_dgrad_nstats)", t_a, 3 * e, 1),
            ("inorm_bwd_stats_stream_kernel + inorm_bwd_stream_kernel (two-pass IN bwd on the same tensor: the path of "
             "norms whose output has a second consumer, i.e. the res-block skip)", t_b, 3 * e, 2)):
        gbs = nbytes / (ms * 1e-3) / 1e9
        out.append({"bound": "hbm", "kernel": name, "achieved": gbs, "peak": hbm_peak, "unit": "GB/s",
                    "frac": gbs / hbm_peak, "ms_per_call": ms, "algorithmic_bytes": nbytes, "launches_per_call": launches})
    return out


DUMP_SAMPLE = 1 << 20       # --dump-outputs: elements kept of a larger output (4 MB in float32; 40 MB for a training step)


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each (name, value) as <out_dir>/<name>.npy, tensors in float32 and Python floats in float64.  A
    tensor of more than DUMP_SAMPLE elements is stored as a fixed seeded sample of its flattened (logical-layout)
    values, the same indices on every run, so that the dumps of two builds compare element for element.  Two runs with
    the same arguments dump identical values: the step adds its fp32 gradient partial sums in a fixed order
    (wgrad_fixup_kernel, colsum_finish_kernel)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays:
        if torch.is_tensor(v):
            v = v.detach().reshape(-1)
            if v.numel() > DUMP_SAMPLE:
                idx = torch.randperm(v.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
                v = v[idx.to(v.device)]
            a = v.float().cpu().numpy()
        else:
            a = np.float64(v)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def step_outputs(model):
    """What a training loop receives from the last optimize_parameters(): the losses, the generated volumes (the
    visuals other than the inputs) and the updated weights of each network (its parameters, concatenated)."""
    import torch
    out = [("loss_" + k, v) for k, v in model.get_current_losses().items()]
    out += [(k, v) for k, v in model.get_current_visuals().items() if not k.startswith("real_")]
    for n in model.model_names:
        out.append(("net_" + n, torch.cat([p.detach().reshape(-1) for p in getattr(model, "net" + n).parameters()])))
    return out


def load_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the roofline kernel, from the committed
    `ncu --set full` capture (profiles/roofline_traffic.json); None when no capture of this kernel exists."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            return json.load(f).get(kernel, {}).get("dram_bytes")
    except Exception:  # noqa: BLE001
        return None


def run_gpu(args):
    import torch
    import torch.distributed as dist

    from mra_gan_b200 import networks3D as N3
    from mra_gan_b200 import ops, parallel
    from mra_gan_b200.models import create_model

    rank, world = parallel.init_distributed()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if args.gpus != world and rank == 0:
        print("warning: --gpus %d but WORLD_SIZE=%d (launch with torchrun for N>1)" % (args.gpus, world), file=sys.stderr)
    per_gpu_batch = args.batch if args.batch else default_batch(world)
    N3.set_default_compute_dtype(torch.bfloat16)
    torch.manual_seed(1234)
    import random
    random.seed(1234 + rank)
    import contextlib
    import io
    unet = args.workload == "unet"
    flop_per_sample = FLOP_PER_SAMPLE_STEP_UNET if unet else FLOP_PER_SAMPLE_STEP
    netG = "unet_128" if unet else "resnet_9blocks"
    with contextlib.redirect_stdout(io.StringIO()):
        model = create_model(make_opt(netG=netG))
        model.setup(make_opt(netG=netG))
    I = ops.impl()
    if world > 1:
        parallel.attach(model)
    use_graphs, launch = launch_mode(world, args.no_graphs)
    if use_graphs:
        model.enable_cuda_graphs(warmup_steps=2)        # the step is replayed as two CUDA graphs after 2 eager steps

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / steps

    def measure(batch, steps, warmup, dump_dir=None):
        """(ms per resident step, ms per end-to-end step, kernels per step, host bytes per step) at one batch size;
        with dump_dir, rank 0 writes the outputs of the last resident step there before the end-to-end steps run."""
        g = torch.Generator().manual_seed(1234 + rank)
        shape = (batch, 1, PATCH, PATCH, PATCH)
        host_A = (torch.rand(shape, generator=g) * 2 - 1).pin_memory()
        host_B = (torch.rand(shape, generator=g) * 2 - 1).pin_memory()
        dev_A, dev_B = host_A.cuda(), host_B.cuda()

        def step_resident():
            model.set_input([dev_A, dev_B])
            model.optimize_parameters()

        def step_e2e():
            model.set_input([host_A, host_B])           # pinned host -> device inside the timed region
            model.optimize_parameters()
            model.get_current_losses()                  # device -> host read of the 8 losses (one transfer)

        for _ in range(max(warmup, int(os.environ.get("MRA_BENCH_MIN_WARMUP", "3")))):   # >= 3: two eager steps + the capture step of
                                                        # the graph replay (the env hook shortens ncu launch-list runs only)
            step_resident()
        launches0 = I.launch_count()
        ms_step = timed(step_resident, steps)
        launches = (I.launch_count() - launches0) // steps
        graphs = getattr(model, "_graphs", None)
        if graphs and graphs.get("launches"):
            launches = graphs["launches"]               # replayed from the captured graphs: count taken at capture
        if dump_dir and rank == 0:
            dump_outputs(dump_dir, step_outputs(model))
        ms_e2e = timed(step_e2e, steps)
        return ms_step, ms_e2e, int(launches), int(host_A.numel() * 4 * 2)

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms_step, ms_e2e, launches, h2d = measure(per_gpu_batch, args.steps, args.warmup, args.dump_outputs)
    clocks = sampler.stop() if sampler else None
    err = I.tc_error()
    if err:
        raise RuntimeError("tensor-core kernel barrier time-out (code %d): the timed steps are invalid" % err)

    global_batch = per_gpu_batch * world
    vox = global_batch * PATCH ** 3 / (ms_step * 1e-3)
    vox_e2e = global_batch * PATCH ** 3 / (ms_e2e * 1e-3)
    if world > 1:
        model._graphs = None                       # graphs holding NCCL nodes must go before the communicator
        import gc
        gc.collect()
        barrier()
        dist.destroy_process_group()
    if rank != 0:
        return 0

    sync_stats = dict(model.grad_sync.stats) if getattr(model, "grad_sync", None) is not None else None
    peaks, peak_src = load_peaks()
    # The roofline kernels are timed ALONE against the burst peaks of MEASURED_PEAKS.json, so they get the condition a
    # burst measurement has: a GPU that is not already throttled by the power cap of the 40+ back-to-back training steps
    # just timed (sw_power_cap is active in every step; the same kernel measured 0.183 ms right after the steps and
    # 0.170 ms from idle on one box).  3 s of idle, then each kernel's own warm-up launches.
    torch.cuda.synchronize()
    time.sleep(3.0)
    k_ms, k_flops = time_dominant_kernel(torch, I, per_gpu_batch)
    norm_roof = time_norm_kernels(torch, I, per_gpu_batch, float(peaks.get("hbm_gbs", 6650.0)))
    achieved = k_flops / (k_ms * 1e-3) / 1e12
    peak = float(peaks.get("bf16_tflops", 1590.0))
    line = {
        "metric": "cyclegan_train_voxels_per_sec", "value": vox, "unit": "voxels/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(world, per_gpu_batch, launch, args.workload),
        "e2e": {"value": vox_e2e, "unit": "voxels/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 8 * 4, "ms_per_step": ms_e2e},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "model_tflops": global_batch * flop_per_sample / (ms_step * 1e-3) / 1e12,
        "roofline": {"bound": "tensor", "kernel": "gather_halo_kernel (Conv3d 256->256 k3 fprop, 34^3->32^3, batch %d)" % per_gpu_batch,
                     "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                     "peak_source": peak_src + " bf16_tflops (burst: kernel timed alone, after 3 s of idle)", "ms_per_launch": k_ms,
                     "algorithmic_flop": k_flops,
                     "traffic": load_traffic("gather_halo_kernel_fprop_b%d" % per_gpu_batch)},
        "roofline_hbm": norm_roof,
        "tc_error_flag": err,
    }
    if sync_stats is not None:
        line["grad_sync"] = dict(sync_stats, fused_wgrad=os.environ.get("MRA_DP_FUSED_WGRAD", "1") == "1",
                                 skip_allreduce=os.environ.get("MRA_DP_SKIP_ALLREDUCE", "0") == "1")
    if world == 1 and not args.no_anchor and not args.batch and not unet:
        # the weak-scaling anchor: the SAME program the N > 1 runs execute (config 3's per-GPU batch and launch mode)
        # on one GPU, so that value(N) / (N * anchor.value) compares like with like
        model._graphs = None
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        a_graphs, a_launch = launch_mode(2, args.no_graphs)
        if a_graphs:
            model.enable_cuda_graphs(warmup_steps=2)
        a_batch = default_batch(2)
        a_ms, a_e2e, a_l, _ = measure(a_batch, max(3, min(args.steps, 10)), 3)
        line["anchor"] = {"what": "this program at the N>1 per-GPU batch on ONE GPU (weak-scaling denominator)",
                          "per_gpu_batch": a_batch, "launch": a_launch, "ms_per_step": a_ms,
                          "value": a_batch * PATCH ** 3 / (a_ms * 1e-3), "unit": "voxels/s",
                          "e2e_value": a_batch * PATCH ** 3 / (a_e2e * 1e-3), "gpu_launches": a_l}
    if not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_block()       # rank 0, after the timed region; the other ranks have exited
    print(json.dumps(line), flush=True)
    return 0


def run_infer(args):
    """BASELINE config 5: the test.py sliding-window path on a synthetic 256 x 256 x 160 volume; a "step" is one whole
    volume.  value = volume voxels / s with the volume resident on the device, e2e = volume handed over from pinned
    host memory and the result read back to the host."""
    import contextlib
    import io

    import torch
    import torch.distributed as dist

    from mra_gan_b200 import networks3D as N3
    from mra_gan_b200 import ops, parallel
    from mra_gan_b200.inference import sliding_window_inference, window_grid
    from mra_gan_b200.models import create_model

    rank, world = parallel.init_distributed()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    N3.set_default_compute_dtype(torch.bfloat16)
    I = ops.impl()
    ck = "/tmp/mra_cfg5_%d" % rank
    os.makedirs(ck + "/cfg5", exist_ok=True)
    opt = make_opt(isTrain=False, model="test", model_suffix="", checkpoints_dir=ck, name="cfg5")
    with contextlib.redirect_stdout(io.StringIO()):
        torch.manual_seed(7)                                  # same weights on every rank
        g = N3.define_G(1, 1, 64, "resnet_9blocks", "instance")
        torch.save({k: v.detach().cpu().contiguous() for k, v in g.state_dict().items()}, ck + "/cfg5/latest_net_G.pth")
        del g
        tm = create_model(opt)
        tm.setup(opt)
    shape, patch, stride = (256, 256, 160), (128, 128, 128), args.stride
    host_vol = (torch.rand(shape, generator=torch.Generator().manual_seed(1234)) * 255).pin_memory()
    dev_vol = host_vol.cuda()
    nwin = len(window_grid(shape, patch, stride, stride))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / steps

    out = {}

    def step_resident():
        out["v"] = sliding_window_inference(tm, dev_vol, patch, stride, stride, rank, world, dtype=torch.bfloat16,
                                            windows_per_pass=args.windows_per_pass)

    def step_e2e():
        r = sliding_window_inference(tm, host_vol, patch, stride, stride, rank, world, dtype=torch.bfloat16,
                                     windows_per_pass=args.windows_per_pass)
        if rank == 0:
            out["h"] = r.cpu()

    for _ in range(max(args.warmup, 1)):
        step_resident()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    l0 = I.launch_count()
    ms = timed(step_resident, args.steps)
    launches = (I.launch_count() - l0) // args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, [("label", out["v"])])
    ms_e2e = timed(step_e2e, args.steps)
    clocks = sampler.stop() if sampler else None
    err = I.tc_error()
    check = batched = None
    if world > 1:
        # (1) the sharding logic: the reference's one-window-per-pass loop sharded over the ranks against this rank running
        # every window -- same kernels on the same batches of 1, so only the order of the fp32 accumulation differs
        sh1 = sliding_window_inference(tm, dev_vol, patch, stride, stride, rank, world, dtype=torch.bfloat16, windows_per_pass=1)
        if rank == 0:
            ref = sliding_window_inference(tm, dev_vol, patch, stride, stride, 0, 1, dtype=torch.bfloat16, windows_per_pass=1)
            check = float((sh1 - ref).abs().max())
            # (2) the timed run groups windows into batches: a sample's convolution results do not depend on its batch
            # mates, but the fp32 partial sums of its InstanceNorm statistics are grouped by the persistent schedule, and
            # this UNTRAINED N(0, 0.02) generator amplifies such last-bit differences (see DESIGN.md 5)
            d = (out["v"] - ref).double()
            batched = {"rel_l2": float(d.norm() / (ref.double() - 127.5).norm()), "max_abs": float(d.abs().max())}
    if world > 1:
        barrier()
        dist.destroy_process_group()
    if rank != 0:
        return 0
    nvox = shape[0] * shape[1] * shape[2]
    my_windows = len(range(0, nwin, world))
    line = {
        "metric": "sliding_window_volume_voxels_per_sec", "value": nvox / (ms * 1e-3), "unit": "voxels/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": WORKLOAD_INFER % (stride, stride, nwin), "volume": list(shape), "window": list(patch),
                   "stride": stride, "windows": nwin, "windows_on_rank0": my_windows,
                   "windows_per_pass": args.windows_per_pass, "parallelism": "windows round-robin over %d rank(s)" % world,
                   "l2": "each window's activations (GBs) >> 126 MB L2", "launch": "eager"},
        "window_voxels_per_sec": nwin * patch[0] ** 3 / (ms * 1e-3),
        "model_tflops": nwin * G_FWD_FLOP_PER_WINDOW / (ms * 1e-3) / 1e12,
        "e2e": {"value": nvox / (ms_e2e * 1e-3), "unit": "voxels/s", "h2d_bytes_per_step": nvox * 4,
                "d2h_bytes_per_step": nvox * 4, "ms_per_step": ms_e2e},
        "gpu_launches": int(launches), "clocks": clocks, "tc_error_flag": err,
        "sharded_vs_single_max_abs": check, "batched_vs_one_window_per_pass": batched,
    }
    print(json.dumps(line), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: 2 on 1 GPU, 4 per GPU on N>1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-anchor", action="store_true", help="skip the batch-4 single-GPU anchor measurement (N=1 only)")
    ap.add_argument("--no-graphs", action="store_true", help="run the step eagerly (no CUDA-graph replay)")
    ap.add_argument("--workload", default="train", choices=["train", "unet", "infer"],
                    help="train = BASELINE configs 2/3 (the headline metric), unet = config 4, infer = config 5")
    ap.add_argument("--stride", type=int, default=32, help="--workload infer: window stride (reference default 32)")
    ap.add_argument("--windows-per-pass", type=int, default=4,
                    help="--workload infer: windows a rank sends through the generator as one batch (1 = the reference's loop)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last resident timed step computed (taken before the end-to-end steps) as "
                         "DIR/<name>.npy (float32; outputs over %d elements as a fixed seeded sample), to compare two "
                         "builds output for output" % DUMP_SAMPLE)
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the GPU arm's outputs; --impl reference has none")
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "infer":
        return run_infer(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
