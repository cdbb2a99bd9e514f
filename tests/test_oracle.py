"""Pin the oracle: (a) against the committed fixtures generated from the reference itself
(oracle/make_golden.py), (b) against the live reference when /root/reference is present."""
import os
import random

import numpy as np
import pytest
import torch

from oracle import functional as OF
from oracle import sliding_window as SW
from oracle.ref_import import import_reference, make_opt, reference_available

# fixtures were produced on the build container's CPU; another host's vector ISA may round
# differently, hence small non-zero tolerances.
TOL = 2e-5


def _load(golden_dir, name):
    return torch.load(os.path.join(golden_dir, name), weights_only=False)


def test_nets_match_golden(golden_dir):
    g = _load(golden_dir, "nets_small.pt")
    r = g["resnet9_ngf8"]
    sd = OF.make_weights(OF.resnet_g_spec(1, 1, 8, 9), r["weight_seed"])
    assert OF.weights_checksum(sd) == pytest.approx(r["checksum"], rel=1e-12)
    x, _ = OF.synthetic_patches(2, 32, seed=r["input_seed"])
    y = OF.resnet_generator(sd, x, 9)
    assert OF.rel_l2(y, r["y"]) < TOL
    assert OF.rel_l2(sd["model.2.running_mean"], r["running_mean_2"]) < TOL
    assert OF.rel_l2(sd["model.2.running_var"], r["running_var_2"]) < TOL
    for sig in (False, True):
        r = g["nlayer3_ndf8_sig%d" % sig]
        sd = OF.make_weights(OF.nlayer_d_spec(1, 8, 3), r["weight_seed"])
        y = OF.nlayer_discriminator(sd, x, 3, use_sigmoid=sig)
        assert y.shape == r["y"].shape == (2, 1, 2, 2, 2)
        assert OF.rel_l2(y, r["y"]) < TOL
    r = g["unet5_ngf8"]
    sd = OF.make_weights(OF.unet_g_spec(1, 1, 5, 8), r["weight_seed"])
    assert OF.rel_l2(OF.unet_generator(sd, x, 5), r["y"]) < TOL


def test_unet7_matches_golden(golden_dir):
    r = _load(golden_dir, "nets_small.pt")["unet7_ngf4"]
    sd = OF.make_weights(OF.unet_g_spec(1, 1, 7, 4), r["weight_seed"], scale=0.2)
    x, _ = OF.synthetic_patches(1, 128, seed=r["input_seed"])
    with torch.no_grad():
        y = OF.unet_generator(sd, x, 7)
    assert OF.rel_l2(y[:, :, ::4, ::4, ::4], r["y_sub"]) < 1e-4
    assert float(y.double().abs().sum()) == pytest.approx(r["y_abs"], rel=1e-4)


@pytest.mark.parametrize("case", ["lsgan", "bce", "lsgan_b2", "unet5"])
def test_cyclegan_step_matches_golden(golden_dir, case):
    r = _load(golden_dir, "cyclegan_step_small.pt")[case]
    random.seed(1234)
    sds = OF.build_cyclegan_weights(r["ngf"], r["ndf"], seed=r["weight_seed"], netG=r["netG"])
    for sd, cs in zip(sds, r["checksums"]):
        assert OF.weights_checksum(sd) == pytest.approx(cs, rel=1e-12)
    m = OF.CycleGANOracle(*sds, netG=r["netG"], no_lsgan=r["no_lsgan"], pool_size=r["pool_size"])
    for st in r["steps"]:
        A, B = OF.synthetic_patches(r["batch"], r["size"], seed=st["input_seed"])
        m.optimize_parameters(A, B)
        got = m.current_losses()
        for k, v in st["losses"].items():
            assert got[k] == pytest.approx(v, rel=2e-4, abs=1e-6), k
        assert float(m.losses["cor_coe_GA"]) == pytest.approx(st["cor_coe_GA"], rel=1e-4)
        assert OF.rel_l2(OF.golden_sample(m.fake_B), st["fake_B"]) < 1e-4
        assert OF.rel_l2(OF.golden_sample(m.rec_A), st["rec_A"]) < 1e-4
        if "grads" in st:
            for key, (nrm, samp) in st["grads"].items():
                net, pk = key.split(".", 1)
                gr = m.sd[net][pk].grad
                assert float(gr.double().norm()) == pytest.approx(nrm, rel=5e-3), key
        with torch.no_grad():
            post = m.G("G_A", A)
        # reference-vs-reference noise floor after an Adam step is ~1e-3..1e-2 max-abs across
        # CPU backends (SURVEY.md section 7-1); same host + same kernels is far tighter.
        assert float((OF.golden_sample(post) - st["post_G_A"]).abs().max()) < 5e-3


def test_sliding_window_matches_golden(golden_dir):
    r = _load(golden_dir, "sliding_window_small.pt")
    sd = OF.make_weights(OF.resnet_g_spec(1, 1, 8, 9), r["weight_seed"], scale=r["weight_scale"])
    assert OF.weights_checksum(sd) == pytest.approx(r["checksum"], rel=1e-12)
    vol = np.random.RandomState(r["vol_seed"]).uniform(0, 255, size=r["shape"]).astype(np.float32)

    def gen(batch):
        with torch.no_grad():
            return OF.resnet_generator(sd, torch.from_numpy(batch), 9, training=True)[0, 0].numpy()

    out = SW.sliding_window_inference(vol, gen, r["patch"], *r["stride"])
    ref = r["label"].numpy()
    assert out.shape == ref.shape == r["shape"]
    assert np.abs(out - ref).max() < 2e-3      # 0..255 scale


def test_window_grid_counts():
    # BASELINE config 5: (256,256,160), 128^3 windows: stride 32 -> 5x5x2, stride 64 -> 3x3x2
    assert len(SW.window_grid((256, 256, 160), (128,) * 3, 32, 32)) == 50
    assert len(SW.window_grid((256, 256, 160), (128,) * 3, 64, 64)) == 18
    g = SW.window_grid((72, 64, 42), (32,) * 3, 16, 16)
    assert len(g) == 4 * 3 * 2 and g[-1] == (40, 72, 32, 64, 10, 42)


def test_lambda_lr_rule():
    # lr constant through epoch 499, linear to 0 at 600 with the defaults (SURVEY.md section 5)
    assert OF.lambda_lr(0, 1, 500, 100) == 1.0
    assert OF.lambda_lr(498, 1, 500, 100) == 1.0
    assert OF.lambda_lr(499, 1, 500, 100) == pytest.approx(1 - 1 / 101)
    assert OF.lambda_lr(599, 1, 500, 100) == pytest.approx(0.0, abs=1e-12)


@pytest.mark.reference
@pytest.mark.skipif(not reference_available(), reason="/root/reference not present")
def test_oracle_vs_live_reference():
    nw, cycle_mod, _, _ = import_reference()
    # key layouts
    for name, spec in (("resnet_9blocks", OF.resnet_g_spec(1, 1, 8, 9)),
                       ("resnet_6blocks", OF.resnet_g_spec(1, 1, 8, 6)),
                       ("unet_custom", OF.unet_g_spec(1, 1, 5, 8)),
                       ("unet_256", OF.unet_g_spec(1, 1, 8, 8))):
        net = nw.define_G(1, 1, 8, name, "instance", False, "normal", 0.02, 0)
        assert [(k, tuple(v.shape)) for k, v in net.state_dict().items()] == list(spec.items())
    with pytest.raises(NotImplementedError):
        nw.define_G(1, 1, 8, "unet_128", "instance")
    net = nw.define_D(1, 8, "n_layers", 3, "instance", False, "normal", 0.02, 0)
    assert [(k, tuple(v.shape)) for k, v in net.state_dict().items()] == list(OF.nlayer_d_spec(1, 8, 3).items())
    # one full step, same weights, same inputs: losses bit-comparable
    opt = make_opt(ngf=8, ndf=8, pool_size=2)
    random.seed(5)
    m = cycle_mod.CycleGANModel()
    m.initialize(opt)
    sds = OF.build_cyclegan_weights(8, 8, seed=77)
    for net, sd in zip((m.netG_A, m.netG_B, m.netD_A, m.netD_B), sds):
        net.load_state_dict({k: v.clone() for k, v in sd.items()})
    random.seed(5)
    o = OF.CycleGANOracle(*OF.build_cyclegan_weights(8, 8, seed=77), pool_size=2)
    for s in range(2):
        A, B = OF.synthetic_patches(1, 32, seed=s)
        m.set_input([A, B])
        m.optimize_parameters()
        o.optimize_parameters(A, B)
        ref = m.get_current_losses()
        got = o.current_losses()
        for k in ref:
            assert got[k] == pytest.approx(ref[k], rel=1e-5, abs=1e-7), (s, k)
