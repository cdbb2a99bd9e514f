"""Generate tests/golden/*.pt by running the UNMODIFIED reference (build container only).

    python -m oracle.make_golden

Weights are synthetic and regenerated from seeds at test time (oracle.functional.make_weights);
each fixture stores a checksum of them, the inputs' seeds and the REFERENCE's outputs (the larger ones as
``OF.golden_sample``).
"""
import os
import random
import sys
import textwrap
from collections import OrderedDict

import numpy as np
import torch

from . import functional as OF
from .ref_import import REFERENCE_ROOT, import_reference, make_opt

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def _load(net, sd):
    net.load_state_dict({k: v.clone() for k, v in sd.items()}, strict=True)
    return net


def gen_nets(nw):
    out = {}
    # resnet_9blocks, ngf=8, 32^3, batch 2
    spec = OF.resnet_g_spec(1, 1, 8, 9)
    sd = OF.make_weights(spec, 11)
    net = _load(nw.define_G(1, 1, 8, "resnet_9blocks", "instance", False, "normal", 0.02, 0), sd)
    assert list(net.state_dict().keys()) == list(spec.keys())
    x, _ = OF.synthetic_patches(2, 32, seed=5)
    y = net(x)
    out["resnet9_ngf8"] = dict(weight_seed=11, input_seed=5, checksum=OF.weights_checksum(sd),
                               y=y.detach().clone(),
                               running_mean_2=net.state_dict()["model.2.running_mean"].clone(),
                               running_var_2=net.state_dict()["model.2.running_var"].clone())
    # 3-layer PatchGAN, ndf=8, 32^3, batch 2, with and without sigmoid
    spec = OF.nlayer_d_spec(1, 8, 3)
    sd = OF.make_weights(spec, 12)
    for sig in (False, True):
        net = _load(nw.define_D(1, 8, "n_layers", 3, "instance", sig, "normal", 0.02, 0), sd)
        assert list(net.state_dict().keys()) == list(spec.keys())
        out["nlayer3_ndf8_sig%d" % sig] = dict(weight_seed=12, input_seed=5,
                                               checksum=OF.weights_checksum(sd),
                                               y=net(x).detach().clone())
    # unet_custom (5 downs), ngf=8, 32^3, batch 2
    spec = OF.unet_g_spec(1, 1, 5, 8)
    sd = OF.make_weights(spec, 13)
    net = _load(nw.define_G(1, 1, 8, "unet_custom", "instance", False, "normal", 0.02, 0), sd)
    assert list(net.state_dict().keys()) == list(spec.keys())
    out["unet5_ngf8"] = dict(weight_seed=13, input_seed=5, checksum=OF.weights_checksum(sd),
                             y=net(x).detach().clone())
    # intended unet_128 (7 downs; dead branch in define_G, networks3D.py:94), ngf=4, 128^3, batch 1
    spec = OF.unet_g_spec(1, 1, 7, 4)
    sd = OF.make_weights(spec, 14, scale=0.2)
    net = _load(nw.UnetGenerator(1, 1, 7, 4, norm_layer=nw.get_norm_layer("instance")), sd)
    assert list(net.state_dict().keys()) == list(spec.keys())
    x7, _ = OF.synthetic_patches(1, 128, seed=6)
    y7 = net(x7).detach()
    out["unet7_ngf4"] = dict(weight_seed=14, input_seed=6, checksum=OF.weights_checksum(sd),
                             y_sub=y7[:, :, ::4, ::4, ::4].clone(), y_sum=float(y7.double().sum()),
                             y_abs=float(y7.double().abs().sum()))
    return out


BN_NETS = {"resnet6_ngf8": ("G", "resnet_6blocks", 21), "nlayer3_ndf8": ("D", "n_layers", 22),
           "unet5_ngf8": ("G", "unet_custom", 23)}


def build_bn_net(mod, kind, which):
    """norm='batch' networks of the fixture, built through either module's define_G / define_D."""
    if kind == "G":
        return mod.define_G(1, 1, 8, which, "batch", False, "normal", 0.02, [])
    return mod.define_D(1, 8, which, 3, "batch", False, "normal", 0.02, [])


def gen_batchnorm(nw):
    """norm='batch' (networks3D.py:17): train-mode forward, backward of mean(y^2), buffers after the step, and an
    eval-mode forward on the updated running statistics (reference modules cast to fp64, results stored as fp32)."""
    out = {}
    x, _ = OF.synthetic_patches(2, 32, seed=7)
    for name, (kind, which, seed) in BN_NETS.items():
        net = build_bn_net(nw, kind, which)
        sd = OF.make_weights_like(net.state_dict(), seed)
        _load(net, sd)
        net.double().train()                               # the reference's modules evaluated in fp64: the 1^3 bottleneck of
        x = x.double()                                     # the UNet (2 values per channel) is ill-conditioned in fp32
        xi = x.clone().requires_grad_(True)
        y = net(xi)
        y.square().mean().backward()
        grads = {k: p.grad.detach().float() for k, p in net.named_parameters()
                 if p.grad is not None and (p.dim() == 1 or k in ("model.1.weight", "model.0.weight", "model.model.0.weight"))}
        bufs = {k: (b.detach().float() if b.is_floating_point() else b.detach().clone()) for k, b in net.named_buffers()}
        net.eval()
        with torch.no_grad():
            y_eval = net(x)
        # the reference's own fp32 run against its fp64 run: the conditioning floor an fp32 implementation sits on
        net32 = _load(build_bn_net(nw, kind, which), sd).train()
        x32 = x.float().requires_grad_(True)
        y32 = net32(x32)
        y32.square().mean().backward()
        g32 = dict(net32.named_parameters())
        floor = dict(y=OF.rel_l2(y32.detach(), y.detach()), dx=OF.rel_l2(x32.grad, xi.grad),
                     grads=max(OF.rel_l2(g32[k].grad, v) for k, v in grads.items() if float(v.norm()) > 1e-12))
        out[name] = dict(weight_seed=seed, input_seed=7, checksum=OF.weights_checksum(sd), keys=list(sd.keys()),
                         y=OF.golden_sample(y.float()), dx=xi.grad[:, :, ::2, ::2, ::2].float(), grads=grads, buffers=bufs,
                         y_eval=OF.golden_sample(y_eval.float()), fp32_floor=floor)
    return out


def gen_step(cycle_mod, no_lsgan, netG="resnet_9blocks", ngf=8, size=32, steps=2, batch=1):
    opt = make_opt(ngf=ngf, ndf=8, no_lsgan=no_lsgan, netG=netG, pool_size=2)
    torch.manual_seed(1234)
    random.seed(1234)
    m = cycle_mod.CycleGANModel()
    m.initialize(opt)
    sds = OF.build_cyclegan_weights(ngf, 8, seed=21, netG=netG)
    for net, sd in zip((m.netG_A, m.netG_B, m.netD_A, m.netD_B), sds):
        _load(net, sd)
    m.schedulers = []
    rec = dict(no_lsgan=no_lsgan, netG=netG, ngf=ngf, ndf=8, size=size, batch=batch, weight_seed=21,
               pool_size=2, checksums=[OF.weights_checksum(sd) for sd in sds], steps=[])
    for s in range(steps):
        A, B = OF.synthetic_patches(batch, size, seed=100 + s)
        m.set_input([A, B])
        m.optimize_parameters()
        with torch.no_grad():
            post = m.netG_A(A)   # train-mode forward, also EMA-updates running stats
        st = dict(input_seed=100 + s, losses=dict(m.get_current_losses()),
                  cor_coe_GA=float(m.loss_cor_coe_GA), cor_coe_GB=float(m.loss_cor_coe_GB),
                  fake_B=OF.golden_sample(m.fake_B), rec_A=OF.golden_sample(m.rec_A),
                  idt_A=OF.golden_sample(m.idt_A), post_G_A=OF.golden_sample(post))
        if s == 0:
            # fp64 "truth" for the post-step generator output (SURVEY.md section 4: compare errors against
            # fp64 instead of demanding agreement with one particular fp32 summation order)
            random_state = random.getstate()
            random.seed(1234)
            o64 = OF.CycleGANOracle(*OF.build_cyclegan_weights(ngf, 8, seed=21, netG=netG, dtype=torch.float64),
                                    netG=netG, no_lsgan=no_lsgan, pool_size=2)
            o64.optimize_parameters(A.double(), B.double())
            with torch.no_grad():
                post64 = o64.G("G_A", A.double())
            random.setstate(random_state)
            st["post_G_A_fp64"] = OF.golden_sample(post64.float())
            st["ref_post_err_vs_fp64"] = float((post.double() - post64).abs().max())
            # gradients left in .grad after the step (G grads from backward_G, D from backward_D_*)
            g = {}
            for nm, net in (("G_A", m.netG_A), ("D_A", m.netD_A)):
                for k, p in net.named_parameters():
                    if k.endswith("weight") and p.grad is not None:
                        g[nm + "." + k] = (float(p.grad.double().norm()),
                                           p.grad.flatten()[:: max(1, p.grad.numel() // 64)][:64].clone())
            st["grads"] = g
        rec["steps"].append(st)
    return rec


def gen_sliding(nw, testm):
    """Runs the reference's OWN lines test.py:96-185 (exec of the file slice) on a synthetic
    (72, 64, 41) volume with 32^3 windows at stride 16 (SURVEY.md 8c recipe)."""
    spec = OF.resnet_g_spec(1, 1, 8, 9)
    sd = OF.make_weights(spec, 31, scale=0.05)
    opt = make_opt(isTrain=False, ngf=8, model="test", model_suffix="")
    torch.manual_seed(7)
    model = testm.TestModel()
    model.initialize(opt)
    _load(model.netG, sd)
    rng = np.random.RandomState(1234)
    vol = rng.uniform(0, 255, size=(72, 64, 41)).astype(np.float32)
    src = open(os.path.join(REFERENCE_ROOT, "test.py")).read().split("\n")
    body = textwrap.dedent("\n".join(src[95:185]))
    import math
    import datetime
    from torch.autograd import Variable
    ns = dict(np=np, math=math, torch=torch, Variable=Variable, datetime=datetime,
              tqdm=lambda it: it, model=model, image_np=vol.copy(),
              label_np=np.zeros_like(vol), batch_size=1, patch_size_x=32, patch_size_y=32,
              patch_size_z=32, stride_inplane=16, stride_layer=16,
              pad_x=72, pad_y=64, pad_z=41)
    import test as ref_test  # noqa: F401  (reference module: provides prepare_batch)
    ns["prepare_batch"] = ref_test.prepare_batch
    saved = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self     # test.py:155 hard-codes .cuda()
    try:
        exec(body, ns)
    finally:
        torch.Tensor.cuda = saved
    return dict(weight_seed=31, weight_scale=0.05, checksum=OF.weights_checksum(sd), vol_seed=1234,
                shape=(72, 64, 41), patch=(32, 32, 32), stride=(16, 16),
                label=torch.from_numpy(np.ascontiguousarray(ns["label_np"])))


def gen_options(nw):
    """define_D('pixel') (PixelDiscriminator, networks3D.py:428-450: three 1x1x1 convolutions) with and without the
    sigmoid, and define_G('unet_256') (8 downs, :92-93; needs a 256^3 input) -- forward and the gradient of mean(y^2)
    with respect to the input, from the unmodified reference."""
    out = {}
    x, _ = OF.synthetic_patches(2, 32, seed=8)
    for sig in (False, True):
        net = nw.define_D(1, 8, "pixel", 3, "instance", sig, "normal", 0.02, 0)
        spec = OrderedDict((k, tuple(v.shape)) for k, v in net.state_dict().items())
        sd = OF.make_weights(spec, 41, scale=0.3)
        _load(net, sd)
        xi = x.clone().requires_grad_(True)
        y = net(xi)
        y.square().mean().backward()
        out["pixel_ndf8_sig%d" % sig] = dict(weight_seed=41, weight_scale=0.3, input_seed=8, keys=list(spec.keys()),
                                             shapes=[tuple(v) for v in spec.values()], checksum=OF.weights_checksum(sd),
                                             y=OF.golden_sample(y), dx=OF.golden_sample(xi.grad),
                                             dw0=net.state_dict(keep_vars=True)["net.0.weight"].grad.detach().clone())
    spec = OF.unet_g_spec(1, 1, 8, 2)
    sd = OF.make_weights(spec, 42, scale=0.2)
    net = _load(nw.define_G(1, 1, 2, "unet_256", "instance", False, "normal", 0.02, 0), sd)
    assert list(net.state_dict().keys()) == list(spec.keys())
    x8, _ = OF.synthetic_patches(1, 256, seed=9)
    with torch.no_grad():
        y8 = net(x8)
    out["unet8_ngf2"] = dict(weight_seed=42, weight_scale=0.2, input_seed=9, checksum=OF.weights_checksum(sd),
                             y_sub=y8[:, :, ::8, ::8, ::8].clone(), y_sum=float(y8.double().sum()),
                             y_abs=float(y8.double().abs().sum()))
    return out


def main():
    torch.set_num_threads(8)
    nw, cycle_mod, testm, _ = import_reference()
    os.makedirs(GOLDEN, exist_ok=True)
    if sys.argv[1:] == ["options"]:                        # regenerate this one fixture only
        torch.save(gen_options(nw), os.path.join(GOLDEN, "options_small.pt"))
        return 0
    if sys.argv[1:] == ["batchnorm"]:                      # regenerate this one fixture only
        torch.save(gen_batchnorm(nw), os.path.join(GOLDEN, "batchnorm_small.pt"))
        return 0
    torch.save(gen_nets(nw), os.path.join(GOLDEN, "nets_small.pt"))
    steps = {"lsgan": gen_step(cycle_mod, no_lsgan=False),
             "bce": gen_step(cycle_mod, no_lsgan=True, steps=1),
             "lsgan_b2": gen_step(cycle_mod, no_lsgan=False, steps=1, batch=2),
             "unet5": gen_step(cycle_mod, no_lsgan=False, netG="unet_custom", steps=1)}
    torch.save(steps, os.path.join(GOLDEN, "cyclegan_step_small.pt"))
    torch.save(gen_sliding(nw, testm), os.path.join(GOLDEN, "sliding_window_small.pt"))
    torch.save(gen_batchnorm(nw), os.path.join(GOLDEN, "batchnorm_small.pt"))
    torch.save(gen_options(nw), os.path.join(GOLDEN, "options_small.pt"))
    for f in sorted(os.listdir(GOLDEN)):
        print(f, os.path.getsize(os.path.join(GOLDEN, f)))


if __name__ == "__main__":
    sys.exit(main())
