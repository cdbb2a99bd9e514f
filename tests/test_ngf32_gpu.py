"""The reference's own configuration -- ngf = ndf = 32 (options/*, the authors' opt.txt) -- on the tensor cores: every
conv of resnet_6blocks, the n-layer and pixel discriminators and unet_custom whose channel counts are multiples of 32
reports tcgen05, the networks match the fp64 oracle against the bf16-storage floor, and one optimize_parameters() at
the reference's defaults (resnet_6blocks, BCE, 64^3, batch 2) matches the oracle port."""
import random
from collections import OrderedDict

import pytest
import torch
import torch.nn.functional as F

from mra_gan_b200 import networks3D as N3
from mra_gan_b200 import ops
from mra_gan_b200.models import create_model
from oracle import functional as OF
from oracle.ref_import import make_opt

import test_models_gpu as TM

pytestmark = pytest.mark.gpu


def _pixel_ref(sd, x):
    """fp64 PixelDiscriminator (networks3D.py): 1x1x1 convs, LeakyReLU, InstanceNorm"""
    y = F.leaky_relu(F.conv3d(x, sd["net.0.weight"], sd["net.0.bias"]), 0.2)
    y = F.conv3d(y, sd["net.2.weight"], sd["net.2.bias"])
    y = F.leaky_relu(OF.instance_norm(y, sd, "net.3"), 0.2)
    return F.conv3d(y, sd["net.5.weight"], sd["net.5.bias"])


def _pixel_spec(ndf):
    s = OrderedDict([("net.0.weight", (ndf, 1, 1, 1, 1)), ("net.0.bias", (ndf,)), ("net.2.weight", (2 * ndf, ndf, 1, 1, 1)),
                     ("net.2.bias", (2 * ndf,))])
    OF._norm_keys(s, "net.3", 2 * ndf)
    s["net.5.weight"], s["net.5.bias"] = (1, 2 * ndf, 1, 1, 1), (1,)
    return s


NETS = {
    # kind: (make net, oracle spec, fp64 forward, convs on the tensor cores, patch edge)
    "resnet": (lambda: N3.define_G(1, 1, 32, "resnet_6blocks", "instance"), lambda: OF.resnet_g_spec(1, 1, 32, 6),
               lambda sd, x: OF.resnet_generator(sd, x, 6), 1 + 2 + 12 + 2 + 1, 16),
    "nlayer": (lambda: N3.define_D(1, 32, "n_layers", 3, "instance"), lambda: OF.nlayer_d_spec(1, 32, 3),
               lambda sd, x: OF.nlayer_discriminator(sd, x, 3), 5, 32),
    "unet": (lambda: N3.define_G(1, 1, 32, "unet_custom", "instance"), lambda: OF.unet_g_spec(1, 1, 5, 32),
             lambda sd, x: OF.unet_generator(sd, x, 5), 10, 32),
    # the last layer (64 -> 1, k1) has one output channel and no (kh, kw) taps to fold: CUDA cores, as at ndf = 64
    "pixel": (lambda: N3.define_D(1, 32, "pixel", 3, "instance"), lambda: _pixel_spec(32), _pixel_ref, 2, 16),
}


@pytest.mark.parametrize("kind", sorted(NETS))
def test_ngf32_network_on_the_tensor_cores(kind):
    N3.set_default_compute_dtype(torch.bfloat16)
    mk, spec, fwd, n_tc, edge = NETS[kind]
    sd = OF.make_weights(spec(), 3, dtype=torch.float64, scale=0.05)
    net = TM._load(mk(), {k: v.float() if v.is_floating_point() else v for k, v in sd.items()})
    I = ops.impl()
    dims = (edge,) * 3
    used = [all(I.conv_uses_tensor_cores(m.geom, 2, dims, torch.bfloat16, w) for w in range(3)) for m in net.conv_modules()]
    assert sum(used) == n_tc, used
    x = torch.randn((2, 1) + dims, generator=torch.Generator().manual_seed(1))
    xin = x.cuda().requires_grad_(True)
    y = net(xin)
    gy = torch.randn(y.shape, generator=torch.Generator().manual_seed(2))
    y.backward(gy.cuda())
    assert I.tc_error() == 0
    for k, v in sd.items():
        if v.is_floating_point() and "running_" not in k:
            v.requires_grad_(True)
    xr = x.double().requires_grad_(True)
    yr = fwd(sd, xr)
    yr.backward(gy.double())
    e_f = OF.rel_l2(y.cpu(), yr)
    e_x = OF.rel_l2(xin.grad.cpu(), xr.grad)
    e_w = max(OF.rel_l2(p.grad.cpu(), sd[k].grad) for k, p in net.named_parameters() if k.endswith("weight"))
    f_f, f_x, f_w = TM._bf16_storage_floor(mk, sd, x, gy, xr.grad, yr)
    print("%s ngf/ndf 32 gpu/floor: fwd %.3e/%.3e dx %.3e/%.3e dw %.3e/%.3e" % (kind, e_f, f_f, e_x, f_x, e_w, f_w))
    assert e_f < 1.5 * f_f + 1e-2 and e_x < 1.5 * f_x + 2e-2 and e_w < 1.5 * f_w + 2e-2


def test_reference_default_step_matches_the_oracle_port(tmp_path):
    """resnet_6blocks + 3-layer PatchGAN, ngf = ndf = 32, BCE (no_lsgan), 64^3 patches at batch 2: one
    optimize_parameters() on the tcgen05 path against the fp32 oracle port with the same weights, inputs and pool RNG."""
    N3.set_default_compute_dtype(torch.bfloat16)
    opt = make_opt(ngf=32, ndf=32, netG="resnet_6blocks", no_lsgan=True, batch_size=2, pool_size=50,
                   checkpoints_dir=str(tmp_path))
    random.seed(4321)
    m = create_model(opt)
    m.setup(opt)
    weights = OF.build_cyclegan_weights(32, 32, n_blocks=6, seed=5)
    for net, sd in zip((m.netG_A, m.netG_B, m.netD_A, m.netD_B), weights):
        TM._load(net, sd)
    I = ops.impl()
    for net in (m.netG_A, m.netD_A):
        assert all(I.conv_uses_tensor_cores(c.geom, 2, (64, 64, 64), torch.bfloat16, w)
                   for c in net.conv_modules() for w in range(3))
    A, B = OF.synthetic_patches(2, 64, seed=900)
    m.set_input([A, B])
    m.optimize_parameters()
    got = m.get_current_losses()
    random.seed(4321)
    o = OF.CycleGANOracle(*OF.build_cyclegan_weights(32, 32, n_blocks=6, seed=5), netG="resnet_6blocks", no_lsgan=True,
                          pool_size=50)
    o.optimize_parameters(A, B)
    want = o.current_losses()
    print("ngf 32 default step losses (bf16 GPU vs fp32 oracle port):", {k: (round(got[k], 4), round(want[k], 4)) for k in want})
    for k in want:
        assert got[k] == pytest.approx(want[k], rel=1.5e-2, abs=1e-3), k        # measured on a B200: <= 0.27 %
    e_fake = OF.rel_l2(m.fake_B.cpu(), o.fake_B.detach())
    e_rec = OF.rel_l2(m.rec_A.cpu(), o.rec_A.detach())
    with torch.no_grad():
        post = m.netG_A(A.cuda()).cpu()
        post_ref = o.G("G_A", A)
    e_post = OF.rel_l2(post, post_ref)
    print("   rel-L2: fake_B %.3e rec_A %.3e, G_A(real_A) after the Adam step %.3e" % (e_fake, e_rec, e_post))
    # measured 2.0e-2 / 6.1e-2 / 9.9e-2 (bf16 storage amplified through the untrained cycle, see
    # test_models_gpu.test_config1_step_matches_the_oracle_port)
    assert e_fake < 4e-2 and e_rec < 2e-1
    assert e_post < 3e-1
    assert I.tc_error() == 0
