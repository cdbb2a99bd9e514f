"""Data-parallel semantics on CPU (gloo, world_size 2): R ranks x batch 1 with bucketed gradient
averaging == one process at batch R (SURVEY.md 8e).  Ops are the CPU oracle implementation."""
import os
import random
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import functional as OF


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _build(tmp):
    from mra_gan_b200 import networks3D as N3
    from mra_gan_b200 import ops
    from mra_gan_b200.models import create_model
    from oracle.ops_ref import RefImpl
    from oracle.ref_import import make_opt
    ops.set_impl(RefImpl(torch.float32))
    N3.set_default_compute_dtype(torch.float32)
    opt = make_opt(ngf=4, ndf=4, pool_size=0, checkpoints_dir=tmp, netG="resnet_6blocks")
    random.seed(7)
    torch.manual_seed(7)
    m = create_model(opt)
    m.setup(opt)
    sds = OF.build_cyclegan_weights(4, 4, n_blocks=6, seed=55)
    for net, sd in zip((m.netG_A, m.netG_B, m.netD_A, m.netD_B), sds):
        net.load_state_dict({k: v.clone() for k, v in sd.items()})
    return m


def _grads(m):
    out = {}
    for name in ("G_A", "G_B", "D_A", "D_B"):
        for k, p in getattr(m, "net" + name).named_parameters():
            if k.endswith("weight"):
                out[name + "." + k] = p.grad.detach().clone()
    return out


def _worker(rank, world, port, tmp, q, fused):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.set_num_threads(2)
    from mra_gan_b200 import parallel
    r, w = parallel.init_distributed("gloo")
    assert (r, w) == (rank, world)
    m = _build(tmp)
    if rank == 1:                                   # attach() must broadcast rank 0's weights
        with torch.no_grad():
            for p in m.netG_A.parameters():
                p.add_(0.5)
    sync = parallel.attach(m, bucket_mb=0.05, fused_wgrad=fused)   # small buckets -> several all-reduces per phase
    assert all(c.fuse_wgrad == fused for c in m.netG_A.conv_modules())
    A, B = OF.synthetic_patches(2, 32, seed=9)
    m.set_input([A[rank:rank + 1], B[rank:rank + 1]])
    m.optimize_parameters()
    losses = m.get_current_losses()
    g = _grads(m)
    q.put((rank, losses, {k: v.numpy() for k, v in g.items()}, dict(sync.stats)))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.timeout(600)
@pytest.mark.parametrize("fused", [False, True], ids=["autograd_accumulate", "fused_wgrad"])
def test_two_rank_gradient_averaging_matches_batch_two(tmp_path, fused, monkeypatch):
    """fused = True: the wgrad kernels add every use of a weight straight into its bucket view and the conv modules
    tell the buckets when a weight is final (MRA_DP_FUSED_WGRAD); every bucket must still go out exactly once, from
    inside the backward pass."""
    world, port = 2, _free_port()
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")     # the ranks run on the CPU also where a GPU is visible
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, str(tmp_path), q, fused)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=500) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    res.sort(key=lambda t: t[0])
    # single process, batch 2
    m = _build(str(tmp_path))
    A, B = OF.synthetic_patches(2, 32, seed=9)
    m.set_input([A, B])
    m.optimize_parameters()
    ref_losses, ref_g = m.get_current_losses(), _grads(m)
    from mra_gan_b200 import ops
    ops.set_impl(None)
    for k in ref_losses:
        mean = 0.5 * (res[0][1][k] + res[1][1][k])
        assert mean == pytest.approx(ref_losses[k], rel=1e-4, abs=1e-6), k
    for k, v in ref_g.items():
        g0, g1 = torch.from_numpy(res[0][2][k]), torch.from_numpy(res[1][2][k])
        assert torch.equal(g0, g1), "ranks must hold identical averaged gradients: " + k
        assert OF.rel_l2(g0, v) < 5e-3, k
    stats = res[0][3]
    assert stats["buckets"] > 4 and stats["allreduce_calls"] == stats["buckets"]
    assert stats["late_launches"] == 0, "every bucket must go out from inside the backward pass (overlap)"


def test_bucket_views_are_256_byte_aligned(tmp_path):
    """Every gradient view starts on a 256-byte boundary of its flat bucket, whatever odd-sized parameters (1-element
    biases of the heads) precede it: the fused-wgrad kernels reduce into these views with 16-byte vector atomics
    (a 4-byte shifted view was a `misaligned address` fault on the GPU at N = 2)."""
    from mra_gan_b200 import ops, parallel
    m = _build(str(tmp_path))
    try:
        sync = parallel.attach(m, bucket_mb=0.05, fused_wgrad=True)
        seen = 0
        for phase in sync.phases.values():
            for b in phase:
                base, end = b.flat.data_ptr(), b.flat.data_ptr() + b.flat.numel() * 4
                assert base % 64 == 0               # CPU allocator: 64 B; the CUDA caching allocator hands out 512 B blocks
                for p in b.params:
                    off = p.grad.data_ptr() - base
                    assert off % 256 == 0 and p.grad.data_ptr() + p.numel() * 4 <= end
                    assert p.grad.stride() == p.stride()
                    seen += 1
        assert seen == sum(1 for n in ("G_A", "G_B", "D_A", "D_B") for _ in getattr(m, "net" + n).parameters())
        assert any(p.numel() == 1 for b in sync.phases["D"] for p in b.params)      # the case that broke alignment
    finally:
        ops.set_impl(None)
