"""Host-logic tests (no GPU): the package's module wiring, fused-program compiler, autograd
formulas, optimiser and checkpoint format, exercised with the op-level oracle installed as the op
implementation (``ops.set_impl(RefImpl())``) and compared with the functional oracle and the
fixtures generated from the reference."""
import os
import random

import pytest
import torch

from mra_gan_b200 import networks3D as N3
from mra_gan_b200 import ops
from mra_gan_b200.models import create_model
from oracle import functional as OF
from oracle.ops_ref import RefImpl
from oracle.ref_import import make_opt


@pytest.fixture(autouse=True)
def oracle_ops():
    prev = ops.set_impl(RefImpl(torch.float32))
    N3.set_default_compute_dtype(torch.float32)
    yield
    ops.set_impl(prev)
    N3.set_default_compute_dtype(torch.bfloat16)


def _load(net, sd):
    net.load_state_dict({k: v.clone() for k, v in sd.items()})
    return net


def test_state_dict_layout_matches_reference_spec():
    for name, spec in (("resnet_9blocks", OF.resnet_g_spec(1, 1, 8, 9)), ("resnet_6blocks", OF.resnet_g_spec(1, 1, 8, 6)),
                       ("unet_custom", OF.unet_g_spec(1, 1, 5, 8)), ("unet_128", OF.unet_g_spec(1, 1, 7, 8)),
                       ("unet_256", OF.unet_g_spec(1, 1, 8, 8))):
        net = N3.define_G(1, 1, 8, name, "instance")
        assert [(k, tuple(v.shape)) for k, v in net.state_dict().items()] == list(spec.items()), name
    net = N3.define_D(1, 8, "n_layers", 3, "instance")
    assert [(k, tuple(v.shape)) for k, v in net.state_dict().items()] == list(OF.nlayer_d_spec(1, 8, 3).items())
    net = N3.define_D(1, 8, "basic", norm="instance")
    assert list(net.state_dict().keys()) == list(OF.nlayer_d_spec(1, 8, 3).keys())
    assert [k for k in N3.define_D(1, 8, "pixel", norm="instance").state_dict() if k.endswith("weight")] == \
        ["net.0.weight", "net.2.weight", "net.5.weight"]
    with pytest.raises(NotImplementedError):
        N3.define_G(1, 1, 8, "no_such_net", "instance")
    with pytest.raises(NotImplementedError):
        N3.define_D(1, 8, "no_such_net", norm="instance")


def test_init_matches_torch_rng_stream():
    """define_G draws the same numbers as the reference's nn.Conv3d construction + init.normal_."""
    import torch.nn as nn
    torch.manual_seed(3)
    net = N3.define_G(1, 1, 4, "resnet_6blocks", "instance")
    torch.manual_seed(3)
    convs = []
    for k, v in OF.resnet_g_spec(1, 1, 4, 6).items():
        if k.endswith(".weight"):
            cls = nn.ConvTranspose3d if k in ("model.16.weight", "model.19.weight") else nn.Conv3d
            convs.append((k, cls(v[1] if cls is nn.Conv3d else v[0], v[0] if cls is nn.Conv3d else v[1], v[2])))
    for k, c in convs:
        nn.init.normal_(c.weight.data, 0.0, 0.02)
    sd = net.state_dict()
    for k, c in convs:
        assert torch.equal(sd[k], c.weight.data), k
        assert float(sd[k.replace("weight", "bias")].abs().sum()) == 0.0


def test_fused_program_of_resnet_generator():
    net = N3.define_G(1, 1, 8, "resnet_9blocks", "instance")
    prog = net.program()
    ops_ = [p[0] for p in prog]
    assert ops_[:3] == ["pad", "conv", "norm"] and ops_.count("pad") == 1      # every other pad is fused
    assert ops_.count("conv") == 1 + 2 + 18 + 2 + 1 and ops_.count("save") == 9
    norms = [p for p in prog if p[0] == "norm"]
    assert [p[4] for p in norms] == [0, 0, 1] + [1, 1] * 8 + [1, 0] + [0, 3]   # halo written by each norm
    assert [p[5] for p in norms] == [False] * 3 + [False, True] * 9 + [False] * 2
    assert prog[-1][0] == "conv" and prog[-1][2] == ops.ACT_TANH
    d = N3.define_D(1, 8, "n_layers", 3, "instance", use_sigmoid=True)
    assert [p[0] for p in d.program()] == ["conv", "conv", "norm", "conv", "norm", "conv", "norm", "conv"]
    assert d.program()[0][2] == ops.ACT_LRELU and d.program()[-1][2] == ops.ACT_SIGMOID


def test_nets_match_golden(golden_dir):
    g = torch.load(os.path.join(golden_dir, "nets_small.pt"), weights_only=False)
    x, _ = OF.synthetic_patches(2, 32, seed=5)
    r = g["resnet9_ngf8"]
    net = _load(N3.define_G(1, 1, 8, "resnet_9blocks", "instance"), OF.make_weights(OF.resnet_g_spec(1, 1, 8, 9), r["weight_seed"]))
    y = net(x)
    assert OF.rel_l2(y, r["y"]) < 1e-5
    assert OF.rel_l2(net.state_dict()["model.2.running_mean"], r["running_mean_2"]) < 1e-5
    assert OF.rel_l2(net.state_dict()["model.2.running_var"], r["running_var_2"]) < 1e-5
    for sig in (False, True):
        r = g["nlayer3_ndf8_sig%d" % sig]
        net = _load(N3.define_D(1, 8, "n_layers", 3, "instance", sig), OF.make_weights(OF.nlayer_d_spec(1, 8, 3), r["weight_seed"]))
        assert OF.rel_l2(net(x), r["y"]) < 1e-5
    r = g["unet5_ngf8"]
    net = _load(N3.define_G(1, 1, 8, "unet_custom", "instance"), OF.make_weights(OF.unet_g_spec(1, 1, 5, 8), r["weight_seed"]))
    assert OF.rel_l2(net(x), r["y"]) < 1e-5


@pytest.mark.parametrize("kind", ["resnet", "unet", "disc"])
def test_gradients_match_oracle_autograd(kind):
    if kind == "resnet":
        spec, mk = OF.resnet_g_spec(1, 1, 4, 6), lambda: N3.define_G(1, 1, 4, "resnet_6blocks", "instance")
        fwd = lambda sd, x: OF.resnet_generator(sd, x, 6)
    elif kind == "unet":
        spec, mk = OF.unet_g_spec(1, 1, 5, 4), lambda: N3.define_G(1, 1, 4, "unet_custom", "instance")
        fwd = lambda sd, x: OF.unet_generator(sd, x, 5)
    else:
        spec, mk = OF.nlayer_d_spec(1, 4, 3), lambda: N3.define_D(1, 4, "n_layers", 3, "instance")
        fwd = lambda sd, x: OF.nlayer_discriminator(sd, x, 3)
    sd = OF.make_weights(spec, 7, dtype=torch.float64, scale=0.1)
    net = _load(mk(), {k: v.float() if v.is_floating_point() else v for k, v in sd.items()})
    x = torch.randn(2, 1, 32, 32, 32, generator=torch.Generator().manual_seed(1))
    xin = x.clone().requires_grad_(True)
    y = net(xin)
    gy = torch.randn(y.shape, generator=torch.Generator().manual_seed(2))
    y.backward(gy)
    for k, v in sd.items():
        if v.is_floating_point() and "running_" not in k:
            v.requires_grad_(True)
    xr = x.double().requires_grad_(True)
    yr = fwd(sd, xr)
    yr.backward(gy.double())
    assert OF.rel_l2(y, yr) < 1e-5
    assert OF.rel_l2(xin.grad, xr.grad) < 1e-4
    for k, p in net.named_parameters():
        if k.endswith("weight"):
            assert OF.rel_l2(p.grad, sd[k].grad) < 2e-4, k
    live = {"resnet": ["model.23.bias"], "disc": ["model.0.bias", "model.11.bias"],
            "unet": ["model.model.3.bias"]}[kind]
    named = dict(net.named_parameters())
    for k in live:
        assert OF.rel_l2(named[k].grad, sd[k].grad) < 2e-4, k


@pytest.mark.parametrize("case", ["lsgan", "bce", "lsgan_b2", "unet5"])
def test_cyclegan_step_matches_golden(golden_dir, case, tmp_path):
    r = torch.load(os.path.join(golden_dir, "cyclegan_step_small.pt"), weights_only=False)[case]
    opt = make_opt(ngf=r["ngf"], ndf=r["ndf"], no_lsgan=r["no_lsgan"], netG=r["netG"], pool_size=r["pool_size"],
                   checkpoints_dir=str(tmp_path))
    random.seed(1234)
    m = create_model(opt)
    m.setup(opt)
    assert m.name() == "CycleGANModel"
    for net, sd in zip((m.netG_A, m.netG_B, m.netD_A, m.netD_B),
                       OF.build_cyclegan_weights(r["ngf"], r["ndf"], seed=r["weight_seed"], netG=r["netG"])):
        _load(net, sd)
    for si, st in enumerate(r["steps"]):
        A, B = OF.synthetic_patches(r["batch"], r["size"], seed=st["input_seed"])
        m.set_input([A, B])
        m.optimize_parameters()
        got = m.get_current_losses()
        assert list(got) == ["D_A", "G_A", "cycle_A", "idt_A", "D_B", "G_B", "cycle_B", "idt_B"]
        # step 0 starts from identical weights; later steps sit on the reference-vs-reference noise
        # floor (Adam's first update ~ lr*sign(g) amplifies 1e-6 gradient noise: SURVEY.md 7-1)
        ltol, atol = (5e-4, 1e-4) if si == 0 else (3e-2, 2e-2)
        for k, v in st["losses"].items():
            assert got[k] == pytest.approx(v, rel=ltol, abs=1e-6), k
        assert float(m.loss_cor_coe_GA) == pytest.approx(st["cor_coe_GA"], rel=10 * ltol)
        assert OF.rel_l2(OF.golden_sample(m.fake_B), st["fake_B"]) < atol
        assert OF.rel_l2(OF.golden_sample(m.rec_A), st["rec_A"]) < atol
        assert OF.rel_l2(OF.golden_sample(m.idt_A), st["idt_A"]) < atol
        if "grads" in st:
            named = {"G_A": dict(m.netG_A.named_parameters()), "D_A": dict(m.netD_A.named_parameters())}
            for key, (nrm, samp) in st["grads"].items():
                net, pk = key.split(".", 1)
                assert float(named[net][pk].grad.double().norm()) == pytest.approx(nrm, rel=5e-3), key
        with torch.no_grad():
            post = m.netG_A(A)
        if si == 0:       # after ONE step (north_star); measured floor here ~2.5e-3, see DESIGN.md
            assert float((OF.golden_sample(post) - st["post_G_A"]).abs().max()) < 1e-2
    assert set(m.get_current_visuals()) == {"real_A", "fake_B", "rec_A", "idt_A", "real_B", "fake_A", "rec_B", "idt_B"}


def test_checkpoint_roundtrip_and_reference_format(tmp_path):
    opt = make_opt(ngf=4, ndf=4, checkpoints_dir=str(tmp_path), name="ck")
    m = create_model(opt)
    m.setup(opt)
    m.save_networks("latest")
    saved = torch.load(os.path.join(str(tmp_path), "ck", "latest_net_G_A.pth"))
    assert list(saved.keys()) == list(OF.resnet_g_spec(1, 1, 4, 9).keys())
    assert all(v.is_contiguous() and v.device.type == "cpu" for v in saved.values())
    before = {k: v.clone() for k, v in m.netG_A.state_dict().items()}
    with torch.no_grad():
        for p in m.netG_A.parameters():
            p.add_(1.0)
    m.load_networks("latest")
    for k, v in m.netG_A.state_dict().items():
        assert torch.equal(v, before[k]), k
    # a checkpoint written the reference's way (plain nn.Module state_dict) loads too, incl. a
    # pre-0.4 file without num_batches_tracked and a DataParallel "module." prefix
    legacy = {("module." + k): v for k, v in saved.items() if not k.endswith("num_batches_tracked")}
    torch.save(legacy, os.path.join(str(tmp_path), "ck", "7_net_G_A.pth"))
    for n in ("G_B", "D_A", "D_B"):
        os.replace(os.path.join(str(tmp_path), "ck", "latest_net_%s.pth" % n), os.path.join(str(tmp_path), "ck", "7_net_%s.pth" % n))
    m.load_networks(7)
    # TestModel loads <epoch>_net_G<suffix>.pth
    os.replace(os.path.join(str(tmp_path), "ck", "latest_net_G_A.pth"), os.path.join(str(tmp_path), "ck", "latest_net_G.pth"))
    topt = make_opt(ngf=4, isTrain=False, model="test", model_suffix="", checkpoints_dir=str(tmp_path), name="ck")
    t = create_model(topt)
    t.setup(topt)
    assert t.name() == "TestModel"
    x, _ = OF.synthetic_patches(1, 16, seed=1)
    t.set_input(x)
    t.test()
    assert tuple(t.get_current_visuals()["fake_B"].shape) == (1, 1, 16, 16, 16)


def test_schedulers_and_lr_rule():
    opt = make_opt(ngf=4, ndf=4, niter=2, niter_decay=2, checkpoints_dir="/tmp/mra_sched")
    m = create_model(opt)
    m.setup(opt)
    lrs = []
    for _ in range(5):
        lrs.append(m.optimizers[0].param_groups[0]["lr"])
        m.update_learning_rate()
    want = [2e-4 * OF.lambda_lr(e, 1, 2, 2) for e in range(5)]
    assert lrs == pytest.approx(want)
    bad = make_opt(lr_policy="nope")
    assert isinstance(N3.get_scheduler(m.optimizers[0], bad), NotImplementedError)   # returned, not raised (:40)


def test_no_cpu_fallback_in_product_path():
    ops.set_impl(None)
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            ops.impl()


def test_dropout_option_builds_runs_and_matches_reference_keys():
    """use_dropout=True (SURVEY.md 8f-1): nn.Dropout(0.5) inside the ResNet blocks / inner UNet blocks
    (networks3D.py:244-245, 332-333).  Same state_dict keys as the reference; stochastic in train mode with the
    1/(1-p) scaling and a matching gradient mask, identity in eval mode."""
    import torch
    from mra_gan_b200 import functional as MF
    from mra_gan_b200 import networks3D as N3
    from mra_gan_b200 import ops
    from oracle import ops_ref as R
    prev = ops.set_impl(R.RefImpl(torch.float32))
    N3.set_default_compute_dtype(torch.float32)
    try:
        from oracle.ref_import import import_reference, reference_available
        # the UNet only gets dropout in its (num_downs - 5) innermost ngf*8 blocks (networks3D.py:281-284): 6 downs, 64^3
        builders = (("resnet_6blocks", 32, lambda M: M.define_G(1, 1, 4, "resnet_6blocks", "instance", True, "normal", 0.02, [])),
                    ("unet6", 64, lambda M: M.UnetGenerator(1, 1, 6, 4, norm_layer=M.get_norm_layer("instance"), use_dropout=True)))
        for name, size, build in builders:
            torch.manual_seed(0)
            net = build(N3)
            keys = list(net.state_dict().keys())
            if reference_available():                      # the build container; the GPU box has no /root/reference
                assert keys == list(build(import_reference()[0]).state_dict().keys())
            x = torch.randn(1, 1, size, size, size)
            net.train()
            torch.manual_seed(1); y1 = net(x)
            torch.manual_seed(2); y2 = net(x)
            assert torch.isfinite(y1).all() and not torch.allclose(y1, y2)
            y1.square().mean().backward()
            assert all(torch.isfinite(p.grad).all() for p in net.parameters() if p.grad is not None)
        # the op itself: scaling, mask reuse in the backward pass
        x = torch.randn(2, 4, 4, 4, 8, requires_grad=True)
        torch.manual_seed(3)
        y = MF.DropoutFn.apply(x, 0.5)
        kept = y != 0
        assert 0.3 < kept.float().mean() < 0.7
        assert torch.allclose(y[kept], 2 * x.detach()[kept])
        y.sum().backward()
        assert torch.equal(x.grad != 0, kept) and torch.allclose(x.grad[kept], torch.full_like(x.grad[kept], 2.0))
    finally:
        ops.set_impl(prev)
        N3.set_default_compute_dtype(torch.bfloat16)
