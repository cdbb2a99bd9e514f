"""norm='batch' (SURVEY.md 8f-1): BatchNorm3d(affine) on the InstanceNorm kernels (functional.BatchNormActPadFn).
CPU: host algebra through the oracle ops against torch.nn.functional.batch_norm and against the reference's own
networks; GPU: the same checks through the CUDA kernels."""
import pytest
import torch
import torch.nn.functional as F

from mra_gan_b200 import functional as MF
from mra_gan_b200 import networks3D as N3
from mra_gan_b200 import ops
from mra_gan_b200.ops import ACT_LRELU, ACT_NONE, ACT_RELU
from oracle import functional as OF
from oracle import ops_ref as R


def _fn_case(dev, dtype, act, pad, with_res, training, seed=0):
    """BatchNormActPadFn vs F.batch_norm -> act -> (+ residual) -> replication pad in fp64."""
    gen = torch.Generator().manual_seed(seed)
    n, d, h, w, c = 3, 6, 5, 8, 16
    x = (torch.randn((n, d, h, w, c), generator=gen) * 1.7 + 0.4)
    gam = torch.randn(c, generator=gen) * 0.5 + 1.0
    gam[3] = -0.7                                           # a negative scale must survive the folded form
    bet = torch.randn(c, generator=gen) * 0.3
    res = torch.randn((n, d + 2, h + 2, w + 2, c), generator=gen) if with_res else None
    gy = torch.randn((n, d + 2 * pad, h + 2 * pad, w + 2 * pad, c), generator=gen)
    rm0, rv0 = torch.randn(c, generator=gen) * 0.1, torch.rand(c, generator=gen) + 0.5
    x, gy = x.to(dtype), gy.to(dtype)
    if res is not None:
        res = res.to(dtype)
    # reference in fp64 on the values as stored
    xr = x.double().permute(0, 4, 1, 2, 3).requires_grad_(True)
    gr, br = gam.double().requires_grad_(True), bet.double().requires_grad_(True)
    rm, rv = rm0.double().clone(), rv0.double().clone()
    y = F.batch_norm(xr, rm, rv, gr, br, training=training, momentum=0.1, eps=1e-5)
    y = F.relu(y) if act == ACT_RELU else (F.leaky_relu(y, 0.2) if act == ACT_LRELU else y)
    rr = None
    if res is not None:
        rr = res.double().permute(0, 4, 1, 2, 3).requires_grad_(True)
        y = y + rr[:, :, 1:-1, 1:-1, 1:-1]
    if pad:
        y = F.pad(y, (pad,) * 6, mode="replicate")
    y.backward(gy.double().permute(0, 4, 1, 2, 3))
    # ours
    mod = N3.BatchNorm3d(c).to(dev)
    mod.train(training)
    with torch.no_grad():
        mod.weight.copy_(gam); mod.bias.copy_(bet); mod.running_mean.copy_(rm0); mod.running_var.copy_(rv0)
    xo = x.to(dev).requires_grad_(True)
    ro = res.to(dev).requires_grad_(True) if res is not None else None
    yo = MF.BatchNormActPadFn.apply(xo, None, ro, mod.weight, mod.bias, mod, act, 0.2, pad, 1)
    yo.backward(gy.to(dev))
    tol = 2e-5 if dtype == torch.float32 else 2e-2
    cl = lambda t: t.permute(0, 2, 3, 4, 1)
    assert OF.rel_l2(yo.detach().cpu().double(), cl(y.detach())) < tol
    assert OF.rel_l2(xo.grad.cpu().double(), cl(xr.grad)) < tol
    assert OF.rel_l2(mod.weight.grad.cpu().double(), gr.grad) < tol
    assert OF.rel_l2(mod.bias.grad.cpu().double(), br.grad) < tol
    if res is not None:
        assert OF.rel_l2(ro.grad.cpu().double(), cl(rr.grad)) < tol
    if training:
        assert OF.rel_l2(mod.running_mean.cpu().double(), rm) < 1e-5 and OF.rel_l2(mod.running_var.cpu().double(), rv) < 1e-5
        assert int(mod.num_batches_tracked) == 1


CASES = [(ACT_RELU, 1, False, True), (ACT_NONE, 1, True, True), (ACT_LRELU, 0, False, True), (ACT_RELU, 0, False, False)]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "act%d_pad%d_res%d_train%d" % c)
def test_batchnorm_fn_cpu(case):
    prev = ops.set_impl(R.RefImpl(torch.float64))
    try:
        _fn_case("cpu", torch.float32, *case)
    finally:
        ops.set_impl(prev)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("case", CASES, ids=lambda c: "act%d_pad%d_res%d_train%d" % c)
def test_batchnorm_fn_gpu(case, dtype):
    _fn_case("cuda", dtype, *case)
    assert ops.impl().tc_error() == 0


def _nets_vs_reference(dev, dtype, tol):
    from oracle.ref_import import import_reference, reference_available
    if not reference_available():
        pytest.skip("needs /root/reference")
    ref_n3 = import_reference()[0]
    N3.set_default_compute_dtype(dtype)
    try:
        for build, size in ((lambda M: M.define_G(1, 1, 8, "resnet_6blocks", "batch", False, "normal", 0.02, []), 32),
                            (lambda M: M.define_D(1, 8, "n_layers", 3, "batch", False, "normal", 0.02, []), 32),
                            (lambda M: M.define_G(1, 1, 8, "unet_custom", "batch", False, "normal", 0.02, []), 32)):
            torch.manual_seed(3)
            ref = build(ref_n3).double()
            ours = build(N3).to(dev)
            assert list(ours.state_dict().keys()) == list(ref.state_dict().keys())
            ours.load_state_dict({k: v.clone().float() if v.is_floating_point() else v.clone() for k, v in ref.state_dict().items()})
            x = torch.randn(2, 1, size, size, size, generator=torch.Generator().manual_seed(4))
            yr = ref(x.double())
            yo = ours(x.to(dev))
            assert OF.rel_l2(yo.detach().cpu().double(), yr.detach()) < tol
            yr.square().mean().backward()
            yo.double().square().mean().backward()
            ro, oo = dict(ref.named_parameters()), dict(ours.named_parameters())
            for k, p in ro.items():
                if p.grad is None or float(p.grad.norm()) < 1e-12:
                    continue
                assert OF.rel_l2(oo[k].grad.detach().cpu().double(), p.grad) < 20 * tol, k
            for k, b in ref.named_buffers():
                if b.is_floating_point():
                    assert OF.rel_l2(dict(ours.named_buffers())[k].cpu().double(), b) < 1e-4, k
    finally:
        N3.set_default_compute_dtype(torch.bfloat16)


def _nets_vs_golden(golden_dir, dev, dtype, tol):
    """The committed fixture (oracle/make_golden.py:gen_batchnorm, generated from the unmodified reference): runs on
    the GPU box, where /root/reference is absent."""
    import os
    from oracle.make_golden import BN_NETS, build_bn_net
    g = torch.load(os.path.join(golden_dir, "batchnorm_small.pt"), weights_only=False)
    N3.set_default_compute_dtype(dtype)
    try:
        for name, (kind, which, seed) in BN_NETS.items():
            r = g[name]
            net = build_bn_net(N3, kind, which).to(dev)
            assert list(net.state_dict().keys()) == r["keys"]
            sd = OF.make_weights_like(net.state_dict(), r["weight_seed"])
            assert OF.weights_checksum(sd) == pytest.approx(r["checksum"], rel=1e-12)
            net.load_state_dict(sd)
            net.train()
            x, _ = OF.synthetic_patches(2, 32, seed=r["input_seed"])
            xi = x.to(dev).requires_grad_(True)
            y = net(xi)
            assert OF.rel_l2(OF.golden_sample(y.detach().cpu()), r["y"]) < tol, name
            y.double().square().mean().backward()
            # gradients: the fixture is the reference in fp64; fp32_floor = the reference's own fp32 run against it (the
            # UNet's 1^3 bottleneck normalises 2 values per channel: 5e-3 on dx in fp32, whoever computes it)
            fl = r["fp32_floor"]
            assert OF.rel_l2(xi.grad.cpu()[:, :, ::2, ::2, ::2], r["dx"]) < max(20 * tol, 3 * fl["dx"]), name
            params = dict(net.named_parameters())
            for k, want in r["grads"].items():
                if float(want.norm()) < 1e-12:
                    continue
                assert OF.rel_l2(params[k].grad.detach().cpu(), want) < max(20 * tol, 3 * fl["grads"]), (name, k)
            bufs = dict(net.named_buffers())
            for k, want in r["buffers"].items():
                if want.is_floating_point():
                    assert OF.rel_l2(bufs[k].cpu(), want) < max(tol, 1e-4), (name, k)
                else:
                    assert int(bufs[k]) == int(want), (name, k)
            net.eval()
            with torch.no_grad():
                ye = net(x.to(dev))
            assert OF.rel_l2(OF.golden_sample(ye.cpu()), r["y_eval"]) < tol, name
    finally:
        N3.set_default_compute_dtype(torch.bfloat16)


def test_batchnorm_networks_match_golden_cpu(golden_dir):
    prev = ops.set_impl(R.RefImpl(torch.float32))
    saved = N3.device
    try:
        N3.device = torch.device("cpu")
        _nets_vs_golden(golden_dir, "cpu", torch.float32, 2e-4)
    finally:
        N3.device = saved
        ops.set_impl(prev)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-4), (torch.bfloat16, 6e-2)], ids=["fp32", "bf16"])     # bf16: storage floor 2.5e-2 (CPU oracle ops with bf16 storage)
def test_batchnorm_networks_match_golden_gpu(golden_dir, dtype, tol):
    _nets_vs_golden(golden_dir, "cuda", dtype, tol)
    assert ops.impl().tc_error() == 0


def test_batchnorm_networks_match_reference_cpu():
    prev = ops.set_impl(R.RefImpl(torch.float32))
    try:
        _nets_vs_reference("cpu", torch.float32, 2e-4)
    finally:
        ops.set_impl(prev)


def test_cyclegan_step_with_batchnorm_matches_reference_cpu(tmp_path):
    """The whole drop-in surface with norm='batch' (the reference's own CycleGANModel on the CPU, same weights, same
    inputs, same host RNG): the eight losses of two optimisation steps."""
    import random
    from mra_gan_b200.models import create_model
    from oracle.ref_import import import_reference, make_opt, reference_available
    if not reference_available():
        pytest.skip("needs /root/reference")
    _, cycle_mod, _, _ = import_reference()
    prev = ops.set_impl(R.RefImpl(torch.float32))
    N3.set_default_compute_dtype(torch.float32)
    try:
        opt = make_opt(ngf=4, ndf=4, pool_size=2, norm="batch", checkpoints_dir=str(tmp_path), gpu_ids=-1)
        random.seed(5)
        torch.manual_seed(5)
        ref = cycle_mod.CycleGANModel()
        ref.initialize(make_opt(ngf=4, ndf=4, pool_size=2, norm="batch", checkpoints_dir=str(tmp_path)))
        ours = create_model(opt)
        ours.setup(opt)
        for name in ("G_A", "G_B", "D_A", "D_B"):
            src = getattr(ref, "net" + name).state_dict()
            getattr(ours, "net" + name).load_state_dict({k: v.clone() for k, v in src.items()})
        for s in range(2):
            A, B = OF.synthetic_patches(2, 32, seed=10 + s)
            random.seed(100 + s)
            ref.set_input([A, B]); ref.optimize_parameters()
            want = ref.get_current_losses()
            random.seed(100 + s)
            ours.set_input([A, B]); ours.optimize_parameters()
            got = ours.get_current_losses()
            for k in want:
                assert got[k] == pytest.approx(want[k], rel=2e-3, abs=1e-5), (s, k, got[k], want[k])
    finally:
        ops.set_impl(prev)
        N3.set_default_compute_dtype(torch.bfloat16)
