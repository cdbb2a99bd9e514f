"""GPU parity of the paths VERDICT r1 listed as CPU-only: the sliding-window inference loop on CUDA (odd-z pad,
clamped last windows) against the fixture made from the reference's own test.py lines and against the numpy
restatement; define_D('pixel') and define_G('unet_256') against fixtures generated from the unmodified reference
(oracle/make_golden.py gen_options)."""
import os
from collections import OrderedDict

import numpy as np
import pytest
import torch

from mra_gan_b200 import inference
from mra_gan_b200 import networks3D as N3
from mra_gan_b200 import ops
from mra_gan_b200.models import create_model
from oracle import functional as OF
from oracle import sliding_window as SW
from oracle.ref_import import make_opt

pytestmark = pytest.mark.gpu
DT = {"fp32": torch.float32, "bf16": torch.bfloat16}


@pytest.fixture(params=["fp32", "bf16"])
def mode(request):
    N3.set_default_compute_dtype(DT[request.param])
    yield request.param
    N3.set_default_compute_dtype(torch.bfloat16)


def _emulator_bf16(build, sd, x, loss):
    """The same network on the CPU oracle ops with bf16 STORAGE between layers: the error floor a bf16 implementation
    sits on (a 1x1x1-conv net is a pointwise function of the input, its InstanceNorm cancels a large mean: bf16
    rounding of the pre-norm activations is amplified; fp32 mode is checked to 1e-4 separately)."""
    from oracle.ops_ref import RefImpl
    prev, saved = ops.set_impl(RefImpl(torch.float32)), N3.device
    try:
        N3.device = torch.device("cpu")
        net = build()
        net.load_state_dict({k: v.clone() for k, v in sd.items()})
        xi = x.clone().requires_grad_(True)
        y = net(xi)
        loss(y).backward()
        return y.detach(), xi.grad, net
    finally:
        N3.device = saved
        ops.set_impl(prev)


def _test_model(tmp_path, sd, ngf):
    ck = os.path.join(str(tmp_path), "sw")
    os.makedirs(ck, exist_ok=True)
    torch.save(sd, os.path.join(ck, "latest_net_G.pth"))
    opt = make_opt(ngf=ngf, isTrain=False, model="test", model_suffix="", checkpoints_dir=str(tmp_path), name="sw")
    m = create_model(opt)
    m.setup(opt)
    return m


def test_sliding_window_on_cuda_matches_reference_fixture(golden_dir, tmp_path, mode):
    """test.py:96-185 executed by the reference on a (72, 64, 41) volume (odd z -> edge pad :98-103; 32^3 windows at
    stride 16 -> last windows clamped :125-138) vs inference.sliding_window_inference on the CUDA kernels."""
    r = torch.load(os.path.join(golden_dir, "sliding_window_small.pt"), weights_only=False)
    sd = OF.make_weights(OF.resnet_g_spec(1, 1, 8, 9), r["weight_seed"], scale=r["weight_scale"])
    model = _test_model(tmp_path, sd, 8)
    vol = np.random.RandomState(r["vol_seed"]).uniform(0, 255, size=r["shape"]).astype(np.float32)
    out = inference.sliding_window_inference(model, torch.from_numpy(vol), r["patch"], *r["stride"], dtype=DT[mode])
    assert out.is_cuda and tuple(out.shape) == tuple(r["shape"])
    err = float((out.cpu() - r["label"]).abs().max())
    print("sliding window (%s): max-abs %.3e on the 0..255 scale" % (mode, err))
    if mode == "fp32":
        assert err < 2e-3
    else:
        assert OF.rel_l2(out.cpu() - 127.5, r["label"] - 127.5) < 4e-2
    # one window per generator pass (the reference's loop) == the default two windows per pass: per-sample statistics
    single = inference.sliding_window_inference(model, torch.from_numpy(vol), r["patch"], *r["stride"], dtype=DT[mode],
                                                windows_per_pass=1)
    assert float((single - out).abs().max()) < 1e-4
    # the sharded run (3 ranks' partial sums merged by hand) equals the single-rank result
    parts = [inference.sliding_window_inference.__wrapped__(model, torch.from_numpy(vol), r["patch"], *r["stride"],
                                                            rank=k, world=3, dtype=DT[mode], _local_only=True) for k in range(3)]
    merged = (sum(p[0] for p in parts) / sum(p[1] for p in parts) + 0.01)[:, :, :r["shape"][2]]
    assert float((merged - out).abs().max()) < (1e-3 if mode == "fp32" else 1e-3)
    assert ops.impl().tc_error() == 0


def test_sliding_window_ngf64_tensor_core_path_matches_numpy_restatement(tmp_path):
    """The BASELINE generator (ngf = 64: every conv on the tcgen05 path) over an odd-z volume with clamped windows,
    against oracle/sliding_window.py driven by the functional oracle generator (train-mode norm, test.py never calls
    eval())."""
    N3.set_default_compute_dtype(torch.bfloat16)
    sd = OF.make_weights(OF.resnet_g_spec(1, 1, 64, 9), 33, scale=0.03)
    model = _test_model(tmp_path, sd, 64)
    vol = np.random.RandomState(5).uniform(0, 255, size=(40, 36, 33)).astype(np.float32)
    patch, stride = (32, 32, 32), (8, 8)          # grid 2 x 2 x 2, every last window clamped, z padded 33 -> 34

    def gen(batch):
        with torch.no_grad():
            return OF.resnet_generator(sd, torch.from_numpy(batch), 9).numpy()[0, 0]

    want = SW.sliding_window_inference(vol, gen, patch, *stride)
    got = inference.sliding_window_inference(model, torch.from_numpy(vol), patch, *stride, dtype=torch.bfloat16).cpu().numpy()
    assert got.shape == want.shape == (40, 36, 33)
    e = OF.rel_l2(torch.from_numpy(got - 127.5), torch.from_numpy(want - 127.5))
    print("ngf64 sliding window bf16 vs fp32 oracle: rel-L2 %.3e" % e)
    assert e < 4e-2
    assert ops.impl().tc_error() == 0


def test_pixel_discriminator_matches_reference(golden_dir, mode):
    g = torch.load(os.path.join(golden_dir, "options_small.pt"), weights_only=False)
    x, _ = OF.synthetic_patches(2, 32, seed=8)
    for sig in (False, True):
        r = g["pixel_ndf8_sig%d" % sig]
        sd = OF.make_weights(OrderedDict(zip(r["keys"], r["shapes"])), r["weight_seed"], scale=r["weight_scale"])
        assert OF.weights_checksum(sd) == r["checksum"]
        net = N3.define_D(1, 8, "pixel", 3, "instance", sig)
        assert list(net.state_dict().keys()) == r["keys"]
        net.load_state_dict({k: v.clone() for k, v in sd.items()})
        xi = x.cuda().requires_grad_(True)
        y = net(xi)
        y.square().mean().backward()
        dw0 = net.state_dict(keep_vars=True)["net.0.weight"].grad.cpu()
        e = (OF.rel_l2(OF.golden_sample(y.detach().cpu()), r["y"]), OF.rel_l2(OF.golden_sample(xi.grad.cpu()), r["dx"]),
             OF.rel_l2(dw0, r["dw0"]))
        if mode == "fp32":
            assert e[0] < 1e-4 and e[1] < 1e-3 and e[2] < 1e-3, e
        else:
            fy, fdx, fnet = _emulator_bf16(lambda: N3.define_D(1, 8, "pixel", 3, "instance", sig), sd, x, lambda t: t.square().mean())
            f = (OF.rel_l2(OF.golden_sample(fy), r["y"]), OF.rel_l2(OF.golden_sample(fdx), r["dx"]),
                 OF.rel_l2(fnet.state_dict(keep_vars=True)["net.0.weight"].grad, r["dw0"]))
            print("pixel D bf16 gpu/floor: y %.3e/%.3e dx %.3e/%.3e dw %.3e/%.3e" % (e[0], f[0], e[1], f[1], e[2], f[2]))
            assert all(a < 1.5 * b + 1e-2 for a, b in zip(e, f)), (e, f)
    assert ops.impl().tc_error() == 0


def test_pixel_discriminator_ndf64_uses_tensor_cores():
    """ndf = 64: the 64 -> 128 1x1x1 convolution is a plain GEMM on the tcgen05 gather kernel (one tap)."""
    N3.set_default_compute_dtype(torch.bfloat16)
    net = N3.define_D(1, 64, "pixel", 3, "instance", False)
    I = ops.impl()
    convs = net.conv_modules()
    assert I.conv_uses_tensor_cores(convs[1].geom, 2, (32, 32, 32), torch.bfloat16, 0)
    sd = OF.make_weights(OrderedDict((k, tuple(v.shape)) for k, v in net.state_dict().items()), 43, scale=0.2)
    net.load_state_dict({k: v.clone() for k, v in sd.items()})
    x, _ = OF.synthetic_patches(2, 32, seed=8)
    xi = x.cuda().requires_grad_(True)
    y = net(xi)
    y.square().mean().backward()
    # oracle: the same three 1x1x1 convolutions in fp64 (networks3D.py:436-446)
    import torch.nn.functional as F
    d = {k: v.double() for k, v in sd.items()}
    xr = x.double().requires_grad_(True)
    h = F.leaky_relu(F.conv3d(xr, d["net.0.weight"], d["net.0.bias"]), 0.2)
    h = F.conv3d(h, d["net.2.weight"], d["net.2.bias"])
    h = F.leaky_relu(F.instance_norm(h, eps=1e-5), 0.2)
    yr = F.conv3d(h, d["net.5.weight"], d["net.5.bias"])
    yr.square().mean().backward()
    fy, fdx, _ = _emulator_bf16(lambda: N3.define_D(1, 64, "pixel", 3, "instance", False), sd, x, lambda t: t.square().mean())
    e = (OF.rel_l2(y.detach().cpu(), yr.detach()), OF.rel_l2(xi.grad.cpu(), xr.grad))
    f = (OF.rel_l2(fy, yr.detach()), OF.rel_l2(fdx, xr.grad))
    print("pixel D ndf64 bf16 gpu/floor: y %.3e/%.3e dx %.3e/%.3e" % (e[0], f[0], e[1], f[1]))
    assert e[0] < 1.5 * f[0] + 1e-2 and e[1] < 1.5 * f[1] + 1e-2, (e, f)
    assert I.tc_error() == 0


def test_unet_256_matches_reference(golden_dir, mode):
    r = torch.load(os.path.join(golden_dir, "options_small.pt"), weights_only=False)["unet8_ngf2"]
    sd = OF.make_weights(OF.unet_g_spec(1, 1, 8, 2), r["weight_seed"], scale=r["weight_scale"])
    assert OF.weights_checksum(sd) == r["checksum"]
    net = N3.define_G(1, 1, 2, "unet_256", "instance")
    net.load_state_dict({k: v.clone() for k, v in sd.items()})
    x, _ = OF.synthetic_patches(1, 256, seed=r["input_seed"])
    with torch.no_grad():
        y = net(x.cuda()).cpu()
    assert tuple(y.shape) == (1, 1, 256, 256, 256)
    assert OF.rel_l2(y[:, :, ::8, ::8, ::8], r["y_sub"]) < (1e-4 if mode == "fp32" else 4e-2)
    if mode == "fp32":
        assert abs(float(y.double().sum()) - r["y_sum"]) < 1e-4 * r["y_abs"]
