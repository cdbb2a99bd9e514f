"""CPU restatement of the reference networks, losses and the CycleGAN step (TEST INFRASTRUCTURE).

Everything here is a *functional* restatement driven by ``state_dict``s with the reference's key
layout, computed with torch's CPU kernels in fp32 (or fp64 when the dicts are double) -- the same
third-party arithmetic (ATen / MKL-DNN, unpinned by the reference: SURVEY.md 8c) that the
reference's ``nn.Module``s call.  Each function cites the reference lines it follows.  It never
imports the reference, so it travels to the GPU box.
"""
import math
import random
from collections import OrderedDict

import torch
import torch.nn.functional as F

EPS = 1e-5          # nn.InstanceNorm3d default eps        (models/networks3D.py:19)
MOMENTUM = 0.1      # nn.InstanceNorm3d default momentum   (models/networks3D.py:19)


# --------------------------------------------------------------------------------------
# Architecture specs: state_dict key -> shape, in the reference's state_dict order.
# --------------------------------------------------------------------------------------
def _norm_keys(spec, prefix, c):
    # InstanceNorm3d(affine=False, track_running_stats=True)  (models/networks3D.py:19)
    spec[prefix + ".running_mean"] = (c,)
    spec[prefix + ".running_var"] = (c,)
    spec[prefix + ".num_batches_tracked"] = ()


def resnet_g_spec(input_nc=1, output_nc=1, ngf=64, n_blocks=9):
    """ResnetGenerator key layout (models/networks3D.py:173-215, 224-263)."""
    s = OrderedDict()
    s["model.1.weight"] = (ngf, input_nc, 7, 7, 7)
    s["model.1.bias"] = (ngf,)
    _norm_keys(s, "model.2", ngf)
    idx = 4
    for i in range(2):
        cin, cout = ngf * 2 ** i, ngf * 2 ** (i + 1)
        s["model.%d.weight" % idx] = (cout, cin, 3, 3, 3)
        s["model.%d.bias" % idx] = (cout,)
        _norm_keys(s, "model.%d" % (idx + 1), cout)
        idx += 3
    dim = ngf * 4
    for i in range(n_blocks):
        p = "model.%d.conv_block" % idx
        s[p + ".1.weight"] = (dim, dim, 3, 3, 3)
        s[p + ".1.bias"] = (dim,)
        _norm_keys(s, p + ".2", dim)
        s[p + ".5.weight"] = (dim, dim, 3, 3, 3)
        s[p + ".5.bias"] = (dim,)
        _norm_keys(s, p + ".6", dim)
        idx += 1
    for i in range(2):
        cin = ngf * 2 ** (2 - i)
        cout = cin // 2
        s["model.%d.weight" % idx] = (cin, cout, 3, 3, 3)     # ConvTranspose3d: (in, out, k,k,k)
        s["model.%d.bias" % idx] = (cout,)
        _norm_keys(s, "model.%d" % (idx + 1), cout)
        idx += 3
    idx += 1                                                  # ReplicationPad3d(3)
    s["model.%d.weight" % idx] = (output_nc, ngf, 7, 7, 7)
    s["model.%d.bias" % idx] = (output_nc,)
    return s


def nlayer_d_spec(input_nc=1, ndf=64, n_layers=3):
    """NLayerDiscriminator key layout (models/networks3D.py:381-425)."""
    s = OrderedDict()
    s["model.0.weight"] = (ndf, input_nc, 4, 4, 4)
    s["model.0.bias"] = (ndf,)
    idx = 2
    nf = 1
    for n in range(1, n_layers):
        nf_prev, nf = nf, min(2 ** n, 8)
        s["model.%d.weight" % idx] = (ndf * nf, ndf * nf_prev, 4, 4, 4)
        s["model.%d.bias" % idx] = (ndf * nf,)
        _norm_keys(s, "model.%d" % (idx + 1), ndf * nf)
        idx += 3
    nf_prev, nf = nf, min(2 ** n_layers, 8)
    s["model.%d.weight" % idx] = (ndf * nf, ndf * nf_prev, 4, 4, 4)
    s["model.%d.bias" % idx] = (ndf * nf,)
    _norm_keys(s, "model.%d" % (idx + 1), ndf * nf)
    idx += 3
    s["model.%d.weight" % idx] = (1, ndf * nf, 4, 4, 4)
    s["model.%d.bias" % idx] = (1,)
    return s


def unet_levels(input_nc, output_nc, num_downs, ngf):
    """(outer_nc, inner_nc, in_nc) per block, outermost first (models/networks3D.py:270-287)."""
    lv = [(output_nc, ngf, input_nc), (ngf, ngf * 2, ngf), (ngf * 2, ngf * 4, ngf * 2),
          (ngf * 4, ngf * 8, ngf * 4)]
    for _ in range(num_downs - 5):
        lv.append((ngf * 8, ngf * 8, ngf * 8))
    lv.append((ngf * 8, ngf * 8, ngf * 8))        # innermost
    return lv


def unet_g_spec(input_nc=1, output_nc=1, num_downs=7, ngf=64):
    """UnetGenerator key layout (models/networks3D.py:270-343).  ``use_bias`` is False everywhere
    except the outermost up-conv because the check compares against InstanceNorm2d (:298-301)."""
    lv = unet_levels(input_nc, output_nc, num_downs, ngf)
    s = OrderedDict()

    def rec(level, prefix):
        outer, inner, cin = lv[level]
        outermost, innermost = level == 0, level == len(lv) - 1
        if outermost:
            s[prefix + ".0.weight"] = (inner, cin, 4, 4, 4)
            rec(level + 1, prefix + ".1.model")
            s[prefix + ".3.weight"] = (inner * 2, outer, 4, 4, 4)
            s[prefix + ".3.bias"] = (outer,)
        elif innermost:
            s[prefix + ".1.weight"] = (inner, cin, 4, 4, 4)
            s[prefix + ".3.weight"] = (inner, outer, 4, 4, 4)
            _norm_keys(s, prefix + ".4", outer)
        else:
            s[prefix + ".1.weight"] = (inner, cin, 4, 4, 4)
            _norm_keys(s, prefix + ".2", inner)
            rec(level + 1, prefix + ".3.model")
            s[prefix + ".5.weight"] = (inner * 2, outer, 4, 4, 4)
            _norm_keys(s, prefix + ".6", outer)

    rec(0, "model.model")
    return s


def make_weights(spec, seed, dtype=torch.float32, scale=0.02):
    """Deterministic synthetic weights for a spec (torch CPU generator; independent of the
    reference's init RNG order).  Biases and running stats are made non-trivial on purpose."""
    g = torch.Generator().manual_seed(seed)
    sd = OrderedDict()
    for k, shp in spec.items():
        if k.endswith("num_batches_tracked"):
            sd[k] = torch.zeros((), dtype=torch.long)
        elif k.endswith("running_var"):
            sd[k] = (1.0 + 0.1 * torch.rand(shp, generator=g)).to(dtype)
        elif k.endswith("running_mean"):
            sd[k] = (0.1 * torch.randn(shp, generator=g)).to(dtype)
        else:
            sd[k] = (scale * torch.randn(shp, generator=g)).to(dtype)
    return sd


def make_weights_like(state_dict, seed, scale=0.05):
    """Deterministic weights for ANY network from the keys / shapes of its state_dict (used for norm='batch' nets,
    whose affine scale must sit near 1: a 1-D '.weight' is a BatchNorm gamma)."""
    spec = OrderedDict((k, tuple(v.shape)) for k, v in state_dict.items())
    sd = make_weights(spec, seed, scale=scale)
    g = torch.Generator().manual_seed(seed + 1000)
    for k, shp in spec.items():
        if k.endswith(".weight") and len(shp) == 1:
            sd[k] = 1.0 + 0.3 * torch.randn(shp, generator=g)
    return sd


def weights_checksum(sd):
    """Order-sensitive fp64 checksum used by fixtures to detect RNG drift."""
    acc = 0.0
    for i, (k, v) in enumerate(sd.items()):
        if v.is_floating_point():
            acc += (i + 1) * float(v.double().sum()) + float(v.double().abs().sum())
    return acc


# --------------------------------------------------------------------------------------
# Layers
# --------------------------------------------------------------------------------------
def instance_norm(x, sd, prefix, training=True):
    """nn.InstanceNorm3d(affine=False, track_running_stats=True) (models/networks3D.py:19).
    Train mode: instance statistics + in-place EMA of the running buffers; eval: running stats."""
    rm, rv = sd.get(prefix + ".running_mean"), sd.get(prefix + ".running_var")
    return F.instance_norm(x, running_mean=rm, running_var=rv, weight=None, bias=None,
                           use_input_stats=training or rm is None, momentum=MOMENTUM, eps=EPS)


def rep_pad(x, p):
    # padding_type='reflect' really instantiates nn.ReplicationPad3d (models/networks3D.py:185,232-235)
    return F.pad(x, (p,) * 6, mode="replicate")


def resnet_generator(sd, x, n_blocks=9, training=True, taps=None):
    """ResnetGenerator.forward (models/networks3D.py:185-220, 229-263).  ``taps`` (optional dict)
    receives named intermediate activations for layer-level parity tests."""
    def tap(name, t):
        if taps is not None:
            taps[name] = t
        return t
    h = F.conv3d(rep_pad(x, 3), sd["model.1.weight"], sd["model.1.bias"])
    tap("c1", h)
    h = F.relu(instance_norm(h, sd, "model.2", training))
    tap("c1_act", h)
    idx = 4
    for i in range(2):
        h = F.conv3d(h, sd["model.%d.weight" % idx], sd["model.%d.bias" % idx], stride=2, padding=1)
        h = F.relu(instance_norm(h, sd, "model.%d" % (idx + 1), training))
        tap("down%d" % i, h)
        idx += 3
    for i in range(n_blocks):
        p = "model.%d.conv_block" % idx
        r = F.conv3d(rep_pad(h, 1), sd[p + ".1.weight"], sd[p + ".1.bias"])
        r = F.relu(instance_norm(r, sd, p + ".2", training))
        r = F.conv3d(rep_pad(r, 1), sd[p + ".5.weight"], sd[p + ".5.bias"])
        r = instance_norm(r, sd, p + ".6", training)
        h = h + r
        tap("block%d" % i, h)
        idx += 1
    for i in range(2):
        h = F.conv_transpose3d(h, sd["model.%d.weight" % idx], sd["model.%d.bias" % idx],
                               stride=2, padding=1, output_padding=1)
        h = F.relu(instance_norm(h, sd, "model.%d" % (idx + 1), training))
        tap("up%d" % i, h)
        idx += 3
    idx += 1
    h = F.conv3d(rep_pad(h, 3), sd["model.%d.weight" % idx], sd["model.%d.bias" % idx])
    return torch.tanh(h)


def nlayer_discriminator(sd, x, n_layers=3, use_sigmoid=False, training=True, taps=None):
    """NLayerDiscriminator.forward (models/networks3D.py:391-425)."""
    h = F.leaky_relu(F.conv3d(x, sd["model.0.weight"], sd["model.0.bias"], stride=2, padding=1), 0.2)
    if taps is not None:
        taps["d0"] = h
    idx = 2
    for n in range(1, n_layers):
        h = F.conv3d(h, sd["model.%d.weight" % idx], sd["model.%d.bias" % idx], stride=2, padding=1)
        h = F.leaky_relu(instance_norm(h, sd, "model.%d" % (idx + 1), training), 0.2)
        if taps is not None:
            taps["d%d" % n] = h
        idx += 3
    h = F.conv3d(h, sd["model.%d.weight" % idx], sd["model.%d.bias" % idx], stride=1, padding=1)
    h = F.leaky_relu(instance_norm(h, sd, "model.%d" % (idx + 1), training), 0.2)
    idx += 3
    h = F.conv3d(h, sd["model.%d.weight" % idx], sd["model.%d.bias" % idx], stride=1, padding=1)
    return torch.sigmoid(h) if use_sigmoid else h


def unet_generator(sd, x, num_downs=7, training=True):
    """UnetGenerator.forward (models/networks3D.py:270-343).  The in-place LeakyReLU at the head of
    every non-outermost block mutates the tensor that is later concatenated, so the skip carries
    LeakyReLU(x), not x (:306,343; SURVEY.md 8a-4)."""
    n_levels = num_downs

    def rec(level, prefix, h):
        outermost, innermost = level == 0, level == n_levels - 1
        if outermost:
            d = F.conv3d(h, sd[prefix + ".0.weight"], None, stride=2, padding=1)
            u = rec(level + 1, prefix + ".1.model", d)
            u = F.conv_transpose3d(F.relu(u), sd[prefix + ".3.weight"], sd[prefix + ".3.bias"],
                                   stride=2, padding=1)
            return torch.tanh(u)
        hs = F.leaky_relu(h, 0.2)                      # what the skip actually carries
        d = F.conv3d(hs, sd[prefix + ".1.weight"], None, stride=2, padding=1)
        if innermost:
            u = F.conv_transpose3d(F.relu(d), sd[prefix + ".3.weight"], None, stride=2, padding=1)
            u = instance_norm(u, sd, prefix + ".4", training)
        else:
            d = instance_norm(d, sd, prefix + ".2", training)
            u = rec(level + 1, prefix + ".3.model", d)
            u = F.conv_transpose3d(F.relu(u), sd[prefix + ".5.weight"], None, stride=2, padding=1)
            u = instance_norm(u, sd, prefix + ".6", training)
        return torch.cat([hs, u], 1)

    return rec(0, "model.model", x)


# --------------------------------------------------------------------------------------
# Losses
# --------------------------------------------------------------------------------------
def gan_loss(pred, target_is_real, use_lsgan=True):
    """GANLoss.__call__ (models/networks3D.py:130-150): MSE (LSGAN) or BCE against the expanded
    scalar label 1.0 / 0.0, mean reduction."""
    target = torch.full_like(pred, 1.0 if target_is_real else 0.0)
    return F.mse_loss(pred, target) if use_lsgan else F.binary_cross_entropy(pred, target)


def cor_coe_loss(y_pred, y_target):
    """Cor_CoeLoss (models/networks3D.py:156-166): 1 - r^2."""
    xv = y_pred - torch.mean(y_pred)
    yv = y_target - torch.mean(y_target)
    r = torch.sum(xv * yv) / (torch.sqrt(torch.sum(xv ** 2)) * torch.sqrt(torch.sum(yv ** 2)))
    return 1 - r ** 2


class ImagePoolRef:
    """ImagePool.query (models/cycle_gan_model.py:8-35); host RNG = python ``random``."""

    def __init__(self, pool_size):
        self.pool_size, self.num_imgs, self.images = pool_size, 0, []

    def query(self, images):
        if self.pool_size == 0:
            return images
        out = []
        for image in images:
            image = image.detach().unsqueeze(0)
            if self.num_imgs < self.pool_size:
                self.num_imgs += 1
                self.images.append(image)
                out.append(image)
            elif random.uniform(0, 1) > 0.5:
                rid = random.randint(0, self.pool_size - 1)
                tmp = self.images[rid].clone()
                self.images[rid] = image
                out.append(tmp)
            else:
                out.append(image)
        return torch.cat(out, 0)


def lambda_lr(epoch, epoch_count, niter, niter_decay):
    """get_scheduler 'lambda' rule (models/networks3D.py:28-32)."""
    return 1.0 - max(0, epoch + 1 + epoch_count - niter) / float(niter_decay + 1)


# --------------------------------------------------------------------------------------
# The CycleGAN optimisation step
# --------------------------------------------------------------------------------------
class CycleGANOracle:
    """Functional restatement of CycleGANModel (models/cycle_gan_model.py:64-240) for the
    resnet-generator + n-layer-discriminator family (and the UNet generator).

    Parameters live in four state_dicts with the reference key layout; Adam is torch's own
    (the reference calls torch.optim.Adam, models/cycle_gan_model.py:107-110).
    """

    def __init__(self, sd_G_A, sd_G_B, sd_D_A, sd_D_B, *, netG="resnet_9blocks", n_layers_D=3,
                 no_lsgan=False, pool_size=50, lr=2e-4, beta1=0.5, lambda_A=10.0, lambda_B=10.0,
                 lambda_identity=0.5, lambda_co_A=2, lambda_co_B=2):
        self.sd = {"G_A": sd_G_A, "G_B": sd_G_B, "D_A": sd_D_A, "D_B": sd_D_B}
        for sd in self.sd.values():
            for k, v in sd.items():
                if v.is_floating_point() and "running_" not in k:
                    v.requires_grad_(True)
        self.netG, self.n_layers_D = netG, n_layers_D
        self.use_lsgan = not no_lsgan
        self.lam = (lambda_A, lambda_B, lambda_identity, lambda_co_A, lambda_co_B)
        self.fake_A_pool, self.fake_B_pool = ImagePoolRef(pool_size), ImagePoolRef(pool_size)
        pg = lambda names: [v for n in names for k, v in self.sd[n].items() if v.requires_grad]
        self.optimizer_G = torch.optim.Adam(pg(["G_A", "G_B"]), lr=lr, betas=(beta1, 0.999))
        self.optimizer_D = torch.optim.Adam(pg(["D_A", "D_B"]), lr=lr, betas=(beta1, 0.999))
        self.losses = OrderedDict()

    # -- nets ---------------------------------------------------------------------------
    def G(self, name, x):
        sd = self.sd[name]
        if self.netG.startswith("resnet"):
            return resnet_generator(sd, x, n_blocks=int(self.netG.split("_")[1][0]))
        downs = {"unet_custom": 5, "unet_128": 7, "unet_256": 8}[self.netG]
        return unet_generator(sd, x, num_downs=downs)

    def D(self, name, x):
        return nlayer_discriminator(self.sd[name], x, self.n_layers_D, use_sigmoid=not self.use_lsgan)

    def _set_requires_grad_D(self, flag):
        for n in ("D_A", "D_B"):
            for k, v in self.sd[n].items():
                if v.is_floating_point() and "running_" not in k:
                    v.requires_grad_(flag)

    # -- step ---------------------------------------------------------------------------
    def forward(self, real_A, real_B):
        # models/cycle_gan_model.py:121-136
        self.real_A, self.real_B = real_A, real_B
        self.fake_B = self.G("G_A", real_A)
        self.rec_A = self.G("G_B", self.fake_B)
        self.fake_A = self.G("G_B", real_B)
        self.rec_B = self.G("G_A", self.fake_A)

    def backward_G(self):
        # models/cycle_gan_model.py:163-225
        lam_A, lam_B, lam_idt, lam_co_A, lam_co_B = self.lam
        L = self.losses
        if lam_idt > 0:
            self.idt_A = self.G("G_A", self.real_B)
            L["idt_A"] = F.l1_loss(self.idt_A, self.real_B) * lam_B * lam_idt
            self.idt_B = self.G("G_B", self.real_A)
            L["idt_B"] = F.l1_loss(self.idt_B, self.real_A) * lam_A * lam_idt
        else:
            L["idt_A"] = L["idt_B"] = 0
        L["G_A"] = gan_loss(self.D("D_A", self.fake_B), True, self.use_lsgan)
        L["G_B"] = gan_loss(self.D("D_B", self.fake_A), True, self.use_lsgan)
        L["cycle_A"] = F.l1_loss(self.rec_A, self.real_A) * lam_A
        L["cycle_B"] = F.l1_loss(self.rec_B, self.real_B) * lam_B
        L["cor_coe_GA"] = cor_coe_loss(self.fake_B, self.real_A) * lam_co_A      # computed, not summed (:217-223)
        L["cor_coe_GB"] = cor_coe_loss(self.fake_A, self.real_B) * lam_co_B
        L["G"] = L["G_A"] + L["G_B"] + L["cycle_A"] + L["cycle_B"] + L["idt_A"] + L["idt_B"]
        L["G"].backward()

    def backward_D_basic(self, name, real, fake):
        # models/cycle_gan_model.py:138-149
        loss_real = gan_loss(self.D(name, real), True, self.use_lsgan)
        loss_fake = gan_loss(self.D(name, fake.detach()), False, self.use_lsgan)
        loss = (loss_real + loss_fake) * 0.5
        loss.backward()
        return loss

    def optimize_parameters(self, real_A, real_B):
        # models/cycle_gan_model.py:227-240
        self.forward(real_A, real_B)
        self._set_requires_grad_D(False)
        self.optimizer_G.zero_grad()
        self.backward_G()
        self.optimizer_G.step()
        self._set_requires_grad_D(True)
        self.optimizer_D.zero_grad()
        self.losses["D_A"] = self.backward_D_basic("D_A", self.real_B, self.fake_B_pool.query(self.fake_B))
        self.losses["D_B"] = self.backward_D_basic("D_B", self.real_A, self.fake_A_pool.query(self.fake_A))
        self.optimizer_D.step()

    def current_losses(self):
        names = ["D_A", "G_A", "cycle_A", "idt_A", "D_B", "G_B", "cycle_B", "idt_B"]
        return OrderedDict((n, float(self.losses[n].detach() if torch.is_tensor(self.losses[n]) else self.losses[n])) for n in names)


def build_cyclegan_weights(ngf, ndf, n_blocks=9, n_layers_D=3, seed=1234, dtype=torch.float32,
                           netG=None):
    """Four deterministic state_dicts (seeds seed, seed+1, seed+2, seed+3)."""
    if netG is None or netG.startswith("resnet"):
        gspec = resnet_g_spec(1, 1, ngf, n_blocks)
    else:
        gspec = unet_g_spec(1, 1, {"unet_custom": 5, "unet_128": 7, "unet_256": 8}[netG], ngf)
    dspec = nlayer_d_spec(1, ndf, n_layers_D)
    return (make_weights(gspec, seed, dtype), make_weights(gspec, seed + 1, dtype),
            make_weights(dspec, seed + 2, dtype), make_weights(dspec, seed + 3, dtype))


def synthetic_patches(batch, size, seed=1234, dtype=torch.float32):
    """U(-1,1) patches, the recipe of SURVEY.md 8(d) config 1."""
    g = torch.Generator().manual_seed(seed)
    shp = (batch, 1) + tuple(size if isinstance(size, (tuple, list)) else (size,) * 3)
    A = torch.rand(shp, generator=g) * 2 - 1
    B = torch.rand(shp, generator=g) * 2 - 1
    return A.to(dtype), B.to(dtype)


def rel_l2(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a - b).norm() / (b.norm() + 1e-300))


def golden_sample(t):
    """What tests/golden/ stores of a network output, flattened: all of it up to 4096 elements, else every 5th element
    (5 is odd, so on the power-of-two extents of the fixtures the sample visits every index of every axis).  This keeps
    each fixture file under 1 MB."""
    t = t.detach().reshape(-1)
    return t if t.numel() <= 4096 else t[::5].clone()
