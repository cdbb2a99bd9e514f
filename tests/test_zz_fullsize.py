"""Parity at BASELINE.json's FULL sizes (config 2: 128^3 patches, batch 2, ngf = ndf = 64, bf16) -- every convolution
of resnet_9blocks and of the 3-layer PatchGAN (SURVEY.md 8a-1: G.c1 .. G.c4, D.1 .. D.5) and the InstanceNorm shapes
between them (8a-2), where the CPU oracle cannot run the whole tensor in seconds.  The convolution family is local and
linear, which gives size-independent checks that still go through the oracle:

* crop parity: an output block depends on a small input crop, so oracle(crop) == kernel(full)[block] for blocks at
  the corners and in the interior of the volume (both samples) -- fprop, dgrad;
* masked wgrad: with the scatter-side operand zero outside a few blocks, the weight gradient of the full-size launch
  equals the sum of the oracle's weight gradients of the crops;
* adjoint identities with dense operands: <conv(x, w), dy> = <x, dgrad(dy, w)> = <w, wgrad(x, dy)>;
* epilogue statistics and bias gradients against sums of the tensors the kernels wrote.

The InstanceNorm + activation + replication-pad kernels are compared with the same composition in torch (fp64, on the
device) over the whole tensor.  Runs last (file name) because it moves the most memory.  The checker itself is pinned on
the CPU: the oracle ops must pass it at small sizes, and an implementation with a deliberate indexing error must not.
Crops and the masked wgrad are bounded element by element (oracle/bounds.py); the adjoint identities and the norm
kernels use BASELINE.json's rel-L2 1e-2 of the bf16 path."""
import pytest
import torch
import torch.nn.functional as F

from mra_gan_b200 import ops
from mra_gan_b200.ops import ACT_LRELU, ACT_NONE, ACT_RELU, ACT_TANH, ConvGeom
from oracle import bounds as B
from oracle import ops_ref as R
from oracle.functional import rel_l2

# name -> (geometry, input dims, activation fused into fprop, epilogue statistics wanted)   [models/networks3D.py]
FULL_LAYERS = {
    "G.c1": (ConvGeom(1, 64, 7, 1, 0), (134,) * 3, ACT_NONE, True),                 # :185-187
    "G.d1": (ConvGeom(64, 128, 3, 2, 1), (128,) * 3, ACT_NONE, True),               # :194-195
    "G.d2": (ConvGeom(128, 256, 3, 2, 1), (64,) * 3, ACT_NONE, True),
    "G.rb": (ConvGeom(256, 256, 3, 1, 0), (34,) * 3, ACT_NONE, True),               # :233,241
    "G.u1": (ConvGeom(256, 128, 3, 2, 1, True, 1), (32,) * 3, ACT_NONE, True),      # :205-208
    "G.u2": (ConvGeom(128, 64, 3, 2, 1, True, 1), (64,) * 3, ACT_NONE, True),
    "G.c4": (ConvGeom(64, 1, 7, 1, 0), (134,) * 3, ACT_TANH, False),                # :211-213
    "D.1": (ConvGeom(1, 64, 4, 2, 1), (128,) * 3, ACT_LRELU, False),                # :392-393
    "D.2": (ConvGeom(64, 128, 4, 2, 1), (64,) * 3, ACT_NONE, True),                 # :402-405
    "D.3": (ConvGeom(128, 256, 4, 2, 1), (32,) * 3, ACT_NONE, True),
    "D.4": (ConvGeom(256, 512, 4, 1, 1), (16,) * 3, ACT_NONE, True),                # :411-414
    "D.5": (ConvGeom(512, 1, 4, 1, 1), (15,) * 3, ACT_NONE, False),                 # :417
}
PATTERNS = [("lo", "lo", "lo"), ("hi", "hi", "hi"), ("mid", "lo", "hi"), ("hi", "mid", "lo")]


def _origin(kind, length, blk):
    far = length - blk
    return {"lo": 0, "hi": far, "mid": min((far // 2) | 1, far)}[kind]      # odd interior origin: all stride-2 parities


def _pad_cl(t, lo, hi):
    """zero-pad (negative = crop) the spatial dims of a channels-last (N, D, H, W, C) tensor; lo / hi per axis."""
    return F.pad(t, (0, 0, lo[2], hi[2], lo[1], hi[1], lo[0], hi[0]))


def _crop(t, n, org, ext):
    return t[n:n + 1, org[0]:org[0] + ext[0], org[1]:org[1] + ext[1], org[2]:org[2] + ext[2]]


def _dot(a, b):
    return float((a.double() * b.double()).sum())


class _Layer:
    """Index algebra shared by the checks.  'Scatter side' = the tensor indexed by o, 'gather side' = the one indexed by
    s*o + t - pad (Conv3d: output / input; ConvTranspose3d: input / output)."""

    def __init__(self, g, dims):
        self.g, self.dims, self.odims = g, tuple(dims), g.out_dims(dims)
        self.S = self.odims if not g.transposed else self.dims
        self.G = self.dims if not g.transposed else self.odims
        s, k, p = g.stride, g.k, g.pad
        self.L = [s * (e - 1) + k for e in self.S]                       # padded gather-side extent
        self.lo = [p] * 3
        self.hi = [self.L[a] - self.G[a] - p for a in range(3)]
        self.g0 = ConvGeom(g.cin, g.cout, k, s, 0, g.transposed, 0)      # same filter, explicit padding
        self.blk = min(min(self.S), k + 1 if s == 1 else 4)
        self.ext = s * (self.blk - 1) + k                                # gather-side extent of one block

    def blocks(self, n):
        for i, pat in enumerate(PATTERNS):
            yield i % n, [_origin(pat[a], self.S[a], self.blk) for a in range(3)]

    def gather_crop(self, padded, n, o0):
        s = self.g.stride
        return _crop(padded, n, [s * o for o in o0], [self.ext] * 3)

    def complete(self, o0):
        """(local slices, global slices) of the gather-side region a scatter-side block determines completely."""
        s, k, p = self.g.stride, self.g.k, self.g.pad
        loc, glo = [], []
        for a in range(3):
            lo = 0 if o0[a] == 0 else k - 1
            hi = self.ext - 1 if o0[a] + self.blk == self.S[a] else s * (self.blk - 1)
            off = s * o0[a] - p                                          # local j -> unpadded index j + off
            lo, hi = max(lo, -off), min(hi, self.G[a] - 1 - off)
            assert hi >= lo
            loc.append(slice(lo, hi + 1))
            glo.append(slice(lo + off, hi + 1 + off))
        return loc, glo


def _acc(I, g, dims, n, dtype, which):
    """accumulation type of op ``which`` of the layer on the route the dispatcher picks (oracle/bounds.py)"""
    import ctypes as C

    from mra_gan_b200 import _lib
    d = _lib.ConvDesc()
    d.n, d.cin, d.cout = n, g.cin, g.cout
    d.din, d.hin, d.win = dims
    d.dout, d.hout, d.wout = g.out_dims(tuple(dims))
    d.k, d.stride, d.pad, d.transposed, d.dtype = g.k, g.stride, g.pad, int(g.transposed), _lib.MRA_BF16
    tc = I.conv_uses_tensor_cores(g, n, dims, dtype, which)
    return B.acc_type(dtype, tc, int(_lib.lib().mra_conv3d_lowering(C.byref(d))) if tc else 0, which)


def check_conv_layer(I, g, dims, n, dtype, dev, tol, act=ACT_NONE, stats=True, seed=0):
    """Every property of the module docstring for one layer; ``I`` is the implementation under test.  Crops and the
    masked wgrad are checked element by element against the fp64 oracle (oracle/bounds.py)."""
    lay = _Layer(g, dims)
    acc = [_acc(I, g, lay.dims, n, dtype, which) for which in range(3)]
    gen = torch.Generator(device=dev).manual_seed(seed)
    rnd = lambda *shape: torch.randn(shape, generator=gen, device=dev)
    x = rnd(n, *lay.dims, g.cin).to(dtype)
    w = (rnd(g.taps, g.cout, g.cin) / (g.taps * g.cin) ** 0.5).to(dtype)
    b = rnd(g.cout)
    cpu = lambda t: t.detach().cpu()
    wc, bc = cpu(w), cpu(b)
    wT = I.pack_weight_t(w, dtype)

    # ---- fprop (+ bias, fused activation, epilogue statistics)
    y, st = I.conv_fprop(x, w, b, g, act=act, slope=0.2, want_stats=stats)
    assert tuple(y.shape) == (n,) + lay.odims + (g.cout,)
    assert bool(torch.isfinite(y.float()).all())
    if stats:
        yd = y.double()
        # the statistics come from the fp32 accumulators, the check sums the STORED tensor: in bf16 the two differ by
        # the rounding of y (2^-9 rms per element), which averages out only over many positions per channel
        npos = lay.odims[0] * lay.odims[1] * lay.odims[2]
        stol = 1e-3 if (dtype != torch.bfloat16 or npos >= 512) else 4e-3
        assert rel_l2(cpu(st[..., 0]), cpu(yd.sum((1, 2, 3)))) < stol, "epilogue sum"
        assert rel_l2(cpu(st[..., 1]), cpu((yd * yd).sum((1, 2, 3)))) < stol, "epilogue sum of squares"
        del yd
    if not g.transposed:
        xpad = _pad_cl(x, lay.lo, lay.hi)
        for ni, o0 in lay.blocks(n):
            pre, mag = B.fprop_ref(lay.gather_crop(xpad, ni, o0), wc, bc, lay.g0)
            B.check_output(_crop(y, ni, o0, [lay.blk] * 3), pre, mag, acc[0], act, 0.2, "fprop n%d %s" % (ni, o0))
    else:
        for ni, i0 in lay.blocks(n):
            pre, mag = B.fprop_ref(_crop(x, ni, i0, [lay.blk] * 3), wc, bc, lay.g0)
            loc, glo = lay.complete(i0)
            sl = (slice(None), loc[0], loc[1], loc[2])
            B.check_output(y[ni:ni + 1, glo[0], glo[1], glo[2]], pre[sl], mag[sl], acc[0], act, 0.2, "fprop n%d %s" % (ni, i0))

    # ---- dgrad
    dy = rnd(n, *lay.odims, g.cout).to(dtype)
    dx = I.conv_dgrad(dy, wT, g, lay.dims)
    assert tuple(dx.shape) == tuple(x.shape)
    wTc = cpu(wT)
    if not g.transposed:
        for ni, o0 in lay.blocks(n):
            want, mag = B.dgrad_ref(_crop(dy, ni, o0, [lay.blk] * 3), wTc, lay.g0, (lay.ext,) * 3)
            loc, glo = lay.complete(o0)
            sl = (slice(None), loc[0], loc[1], loc[2])
            B.check_output(dx[ni:ni + 1, glo[0], glo[1], glo[2]], want[sl], mag[sl], acc[1], what="dgrad n%d %s" % (ni, o0))
    else:
        dypad = _pad_cl(dy, lay.lo, lay.hi)
        for ni, i0 in lay.blocks(n):
            want, mag = B.dgrad_ref(lay.gather_crop(dypad, ni, i0), wTc, lay.g0, (lay.blk,) * 3)
            B.check_output(_crop(dx, ni, i0, [lay.blk] * 3), want, mag, acc[1], what="dgrad n%d %s" % (ni, i0))

    # ---- wgrad with the scatter-side operand zero outside the blocks
    scat = dy if not g.transposed else x
    masked = torch.zeros_like(scat)
    gpad = xpad if not g.transposed else dypad
    dw_want = torch.zeros((g.taps, g.cout, g.cin), dtype=torch.float64)
    dw_mag = torch.zeros_like(dw_want)
    for ni, o0 in lay.blocks(n):
        blk = _crop(scat, ni, o0, [lay.blk] * 3)
        _crop(masked, ni, o0, [lay.blk] * 3).add_(blk)                  # overlapping blocks count twice on both sides
        xa, da = (lay.gather_crop(gpad, ni, o0), blk) if not g.transposed else (blk, lay.gather_crop(gpad, ni, o0))
        want, mag = B.wgrad_ref(xa, da, lay.g0)
        dw_want += want
        dw_mag += mag
    xm, dm = (x, masked) if not g.transposed else (masked, dy)
    dw, db = I.conv_wgrad(xm, dm, g, want_bias=True)
    B.check_elements(dw, dw_want, B.CU[acc[2]] * dw_mag, "masked wgrad", B.W_NAMES)
    B.check_dbias(db, dm, "bias gradient")
    del masked, gpad, xm, dm

    # ---- adjoint identities with dense, correlated operands (so that the inner products are far from zero)
    y0, _ = I.conv_fprop(x, w, None, g)
    dyc = (0.5 * y0.float() + 0.5 * y0.float().std() * rnd(*y0.shape)).to(dtype)
    a = _dot(y0, dyc)
    dxc = I.conv_dgrad(dyc, wT, g, lay.dims)
    dwc, _ = I.conv_wgrad(x, dyc, g, want_bias=False)
    assert a > 0
    assert abs(_dot(x, dxc) - a) < 0.2 * tol * a, ("adjoint dgrad", _dot(x, dxc), a)
    assert abs(_dot(w, dwc) - a) < 0.2 * tol * a, ("adjoint wgrad", _dot(w, dwc), a)


# ------------------------------------------------------------------------------------------------------------------
# the checker on the CPU (small sizes): oracle ops pass, a broken implementation does not
# ------------------------------------------------------------------------------------------------------------------
SMALL = [
    (ConvGeom(3, 5, 3, 1, 0), (9, 8, 10)),
    (ConvGeom(4, 6, 3, 2, 1), (12, 11, 13)),
    (ConvGeom(2, 3, 4, 2, 1), (10, 12, 10)),
    (ConvGeom(3, 4, 4, 1, 1), (7, 8, 9)),
    (ConvGeom(1, 4, 7, 1, 0), (15, 14, 16)),
    (ConvGeom(4, 3, 3, 2, 1, True, 1), (6, 5, 7)),
    (ConvGeom(3, 2, 4, 2, 1, True, 0), (5, 6, 5)),
]


@pytest.mark.parametrize("case", SMALL, ids=lambda c: "c%d-%d_k%d_s%d_p%d_%s" % (c[0].cin, c[0].cout, c[0].k, c[0].stride, c[0].pad, "T" if c[0].transposed else "C"))
def test_checker_accepts_the_oracle(case):
    g, dims = case
    ref = R.RefImpl(torch.float64)
    check_conv_layer(ref, g, dims, 2, torch.float64, "cpu", 1e-6, act=ACT_NONE, stats=True)
    check_conv_layer(ref, g, dims, 1, torch.float64, "cpu", 1e-6, act=ACT_LRELU, stats=False, seed=1)


class _Shifted(R.RefImpl):
    """an implementation with a one-voxel indexing error in one op"""

    def __init__(self, which):
        super().__init__(torch.float64)
        self.which = which

    def conv_fprop(self, *a, **k):
        y, st = super().conv_fprop(*a, **k)
        return (torch.roll(y, 1, 3) if self.which == "fprop" else y), st

    def conv_dgrad(self, *a, **k):
        dx = super().conv_dgrad(*a, **k)
        return torch.roll(dx, 1, 1) if self.which == "dgrad" else dx

    def conv_wgrad(self, *a, **k):
        dw, db = super().conv_wgrad(*a, **k)
        return (torch.roll(dw, 1, 0) if self.which == "wgrad" else dw), db


@pytest.mark.parametrize("which", ["fprop", "dgrad", "wgrad"])
@pytest.mark.parametrize("case", [SMALL[1], SMALL[5]], ids=["conv", "convT"])
def test_checker_rejects_an_indexing_error(case, which):
    g, dims = case
    with pytest.raises(AssertionError):
        check_conv_layer(_Shifted(which), g, dims, 2, torch.float64, "cpu", 1e-6)


# ------------------------------------------------------------------------------------------------------------------
# the CUDA kernels at full size
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FULL_LAYERS))
def test_conv_full_size(name):
    g, dims, act, stats = FULL_LAYERS[name]
    I = ops.impl()
    for which in range(3):
        assert I.conv_uses_tensor_cores(g, 2, dims, torch.bfloat16, which), "tcgen05 path expected"
    check_conv_layer(I, g, dims, 2, torch.bfloat16, "cuda", 1e-2, act=act, stats=stats)
    assert I.tc_error() == 0
    torch.cuda.empty_cache()


# UNet-7 (= the intended unet_128, BASELINE config 4) at ngf = 64 on a 128^3 patch: models/networks3D.py:270-343.
# 7 x Conv3d(k4, s2, p1, no bias) 128^3 -> 1^3 and 7 x ConvTranspose3d(k4, s2, p1) back (VERDICT r1 row 13).
UNET7_LAYERS = {
    "U.d1": (ConvGeom(1, 64, 4, 2, 1), (128,) * 3, ACT_NONE, False),              # outermost down: no norm (:312-314)
    "U.d2": (ConvGeom(64, 128, 4, 2, 1), (64,) * 3, ACT_NONE, True),
    "U.d3": (ConvGeom(128, 256, 4, 2, 1), (32,) * 3, ACT_NONE, True),
    "U.d4": (ConvGeom(256, 512, 4, 2, 1), (16,) * 3, ACT_NONE, True),
    "U.d5": (ConvGeom(512, 512, 4, 2, 1), (8,) * 3, ACT_NONE, True),
    "U.d6": (ConvGeom(512, 512, 4, 2, 1), (4,) * 3, ACT_NONE, True),
    "U.d7": (ConvGeom(512, 512, 4, 2, 1), (2,) * 3, ACT_RELU, False),             # innermost: 2^3 -> 1^3, ReLU, no norm (:319-321)
    "U.u7": (ConvGeom(512, 512, 4, 2, 1, True, 0), (1,) * 3, ACT_NONE, True),     # innermost up: 1^3 -> 2^3
    "U.u6": (ConvGeom(1024, 512, 4, 2, 1, True, 0), (2,) * 3, ACT_NONE, True),
    "U.u5": (ConvGeom(1024, 512, 4, 2, 1, True, 0), (4,) * 3, ACT_NONE, True),
    "U.u4": (ConvGeom(1024, 256, 4, 2, 1, True, 0), (8,) * 3, ACT_NONE, True),
    "U.u3": (ConvGeom(512, 128, 4, 2, 1, True, 0), (16,) * 3, ACT_NONE, True),
    "U.u2": (ConvGeom(256, 64, 4, 2, 1, True, 0), (32,) * 3, ACT_NONE, True),
    "U.u1": (ConvGeom(128, 1, 4, 2, 1, True, 0), (64,) * 3, ACT_TANH, False),     # outermost up (+ bias, Tanh) (:312-316)
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(UNET7_LAYERS))
def test_unet7_conv_full_size(name):
    g, dims, act, stats = UNET7_LAYERS[name]
    I = ops.impl()
    for which in range(3):
        assert I.conv_uses_tensor_cores(g, 2, dims, torch.bfloat16, which), "tcgen05 path expected"
    check_conv_layer(I, g, dims, 2, torch.bfloat16, "cuda", 1e-2, act=act, stats=stats)
    assert I.tc_error() == 0
    torch.cuda.empty_cache()


FULL_NORMS = [
    # n, d, c, pad, act, residual pad            site (models/networks3D.py)
    (2, 128, 64, 0, ACT_RELU, -1),             # :188-189 after G.c1
    (2, 128, 64, 3, ACT_RELU, -1),             # :209-211 after G.u2, ReplicationPad3d(3) of the head
    (2, 64, 128, 0, ACT_RELU, -1),             # :196-197
    (2, 32, 256, 1, ACT_RELU, -1),             # :233-243 inside a res-block
    (2, 32, 256, 1, ACT_NONE, 1),              # :257,262 second norm of a block + skip, padded for the next block
    (2, 32, 128, 0, ACT_LRELU, -1),            # :404-405 D.2
    (2, 15, 512, 0, ACT_LRELU, -1),            # :413-414 D.4
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", FULL_NORMS, ids=lambda c: "n%d_%d^3_c%d_pad%d_act%d_res%d" % c)
def test_inorm_act_pad_full_size(case):
    n, d, c, pad, act, rp = case
    I = ops.impl()
    gen = torch.Generator(device="cuda").manual_seed(2)
    x = (torch.randn((n, d, d, d, c), generator=gen, device="cuda") * 1.5 + 0.3).bfloat16()
    res = torch.randn((n,) + (d + 2 * rp,) * 3 + (c,), generator=gen, device="cuda").bfloat16() if rp >= 0 else None
    gy = torch.randn((n,) + (d + 2 * pad,) * 3 + (c,), generator=gen, device="cuda").bfloat16()
    rm, rv = torch.zeros(c, device="cuda"), torch.ones(c, device="cuda")
    st = I.inorm_stats(x)
    y, mean, rstd = I.inorm_fwd(x, st, res, pad, act, 0.2, rp, running_mean=rm, running_var=rv)
    dx, dres = I.inorm_bwd(gy, x, mean, rstd, pad, act, 0.2, rp)
    # the same composition in torch, fp64, on the values as stored
    cf = lambda t: t.double().permute(0, 4, 1, 2, 3)
    xr = cf(x).requires_grad_(True)
    rm_r, rv_r = torch.zeros(c, device="cuda", dtype=torch.float64), torch.ones(c, device="cuda", dtype=torch.float64)
    yr = F.instance_norm(xr, rm_r, rv_r, use_input_stats=True, momentum=0.1, eps=1e-5)
    yr = F.relu(yr) if act == ACT_RELU else (F.leaky_relu(yr, 0.2) if act == ACT_LRELU else yr)
    rr = None
    if res is not None:
        rr = cf(res).requires_grad_(True)
        yr = yr + rr[:, :, rp:rp + d, rp:rp + d, rp:rp + d]
    if pad:
        yr = F.pad(yr, (pad,) * 6, mode="replicate")
    yr.backward(cf(gy))
    cl = lambda t: t.permute(0, 2, 3, 4, 1)
    assert rel_l2(y.double(), cl(yr.detach())) < 1e-2
    assert rel_l2(dx.double(), cl(xr.grad)) < 1e-2
    if res is not None:
        assert rel_l2(dres.double(), cl(rr.grad)) < 1e-2
    assert rel_l2(rm.double(), rm_r) < 1e-5 and rel_l2(rv.double(), rv_r) < 1e-5
    m_ref = xr.detach().mean((2, 3, 4))
    assert rel_l2(mean.double(), m_ref) < 1e-5
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_generator_forward_full_size_window():
    """One 128^3 window through resnet_9blocks (ngf = 64, bf16, every conv on the tcgen05 path) against the CPU oracle in
    fp32 (~10 s of host time): the unit of work of config 5 and the forward pass of config 2, end to end.  The bf16
    storage floor of this network (CPU oracle ops with bf16 storage) is 1.66e-2 at 32^3 and 64^3 alike; a wrong
    InstanceNorm statistic anywhere in the 19 norms moves the result by tens of percent."""
    from mra_gan_b200 import networks3D as N3
    from oracle import functional as OF
    N3.set_default_compute_dtype(torch.bfloat16)
    sd = OF.make_weights(OF.resnet_g_spec(1, 1, 64, 9), 3, scale=0.03)
    sd["model.26.weight"] = sd["model.26.weight"] * 0.1            # keeps the tanh head out of saturation
    net = N3.define_G(1, 1, 64, "resnet_9blocks", "instance")
    net.load_state_dict({k: v.clone() for k, v in sd.items()})
    x, _ = OF.synthetic_patches(1, 128, seed=9)
    with torch.no_grad():
        y = net(x.cuda()).float().cpu()
        want = OF.resnet_generator(sd, x, 9)
    assert ops.impl().tc_error() == 0
    err = rel_l2(y, want)
    print("resnet_9blocks ngf=64, 128^3 window, bf16 vs fp32 oracle: rel-L2 %.3e (bf16 storage floor 1.66e-2)" % err)
    assert err < 4e-2
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_halo_tail_items_share_a_sample_with_full_tiles():
    """The scheduling case behind the statistics bug fixed in conv_tc_halo.cuh, at a size that runs in a blink: one sample
    of 256 -> 256 channels with 80 CTA-pair tiles on 74 pairs, so the last 6 tiles are split into half-width items and
    12 CTAs process a full-width tile AND a half-width item of the same sample (even units without a channel-base change
    in between).  Statistics, crops (the far corner lies in the split tiles), masked wgrad and adjoints all apply."""
    g, dims = ConvGeom(256, 256, 3, 1, 0), (42, 34, 18)
    I = ops.impl()
    check_conv_layer(I, g, dims, 1, torch.bfloat16, "cuda", 1e-2, stats=True)
    assert I.tc_error() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("n,dims", [(1, (42, 34, 18)), (2, (34, 34, 34)), (27, (4, 34, 18))])
def test_halo_statistics_stay_inside_their_buffer(n, dims):
    """Memory-safety canary for the epilogue statistics of gather_halo_kernel (VERDICT r1 weak #1): the [N][Cn][2] fp64
    block handed to mra_conv3d_fprop sits inside a larger buffer whose other words hold -0.0 -- a stray
    ``atomicAdd(+0.0)`` turns that into +0.0, a stray real sum into anything else -- and every sample's sums must
    equal the sums of the stored output (so nothing leaked into the NEXT sample's rows either).  (2, 34^3) is the
    bench's G.rb launch: 256 pair tiles on 74 pairs, the last 34 split, the split falling inside the last sample;
    (27, 4 x 34 x 18) has 108 tiles of 4 per sample, the last 34 split across samples 18..26."""
    import ctypes as C

    from mra_gan_b200 import _lib
    I = ops.impl()
    g = ConvGeom(256, 256, 3, 1, 0)
    gen = torch.Generator().manual_seed(7)
    x = torch.randn((n,) + dims + (256,), generator=gen).to(torch.bfloat16).cuda()
    w = (torch.randn((27, 256, 256), generator=gen) * 0.02).to(torch.bfloat16).cuda()
    out_dims = g.out_dims(dims)
    y = torch.empty((n,) + out_dims + (256,), dtype=torch.bfloat16, device="cuda")
    words, guard = n * 256 * 2, 4096
    neg0 = torch.tensor([-0.0], dtype=torch.float64).view(torch.int64).item()
    buf = torch.full((guard + words + guard,), -0.0, dtype=torch.float64, device="cuda")
    stats = buf[guard:guard + words]
    d = I._conv_desc(g, n, dims, out_dims, _lib.MRA_BF16)
    _lib.check(I.L.mra_conv3d_fprop(C.byref(d), C.c_void_p(x.data_ptr()), C.c_void_p(w.data_ptr()), None,
                                    C.c_void_p(y.data_ptr()), C.c_void_p(stats.data_ptr()), None, 0, I._stream()),
               "mra_conv3d_fprop")
    torch.cuda.synchronize()
    assert I.tc_error() == 0
    bits = buf.view(torch.int64)
    assert bool((bits[:guard] == neg0).all()), "statistics flush wrote BEFORE its buffer"
    assert bool((bits[guard + words:] == neg0).all()), "statistics flush wrote PAST its buffer"
    # per-sample sums against the stored tensor (bf16-rounded output vs fp32 accumulators: loose on purpose, a leaked
    # or lost tile is a >= 1/256 effect on sum of squares)
    yf = y.double()
    s1 = yf.sum(dim=(1, 2, 3))
    s2 = (yf * yf).sum(dim=(1, 2, 3))
    got = stats.view(n, 256, 2)
    assert float((got[..., 1] - s2).abs().max() / s2.abs().max()) < 2e-3
    assert float((got[..., 0] - s1).abs().max() / s2.sqrt().max()) < 2e-2
