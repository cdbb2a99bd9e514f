"""The whole range the conv dispatcher sends to the tensor cores (mra_conv3d_uses_tensor_cores: csrc/conv_tc.cuh
gather_eligible / wgrad_eligible, csrc/conv_special.cuh stem / head / im2col / ConvTranspose3d(C -> 1) lowerings),
not only the layer shapes of the three networks: channel counts 64 .. 512 on both sides (n tiles of 64 / 128 / 256,
3 or 5 of them, ragged second m tile at 192), k = 1 .. 4 with every padding, stride 1 and 2, ConvTranspose3d with and
without output padding, odd / prime / unit extents, w lines longer than a box, batches 1, 2, 3 and 5 (tiles and
stream-K ranges across sample boundaries), wgrad items shared between CTAs (fix-up kernel) or not, CTA pairs, and the
lowerings at widths up to 256.  Every output element is checked against the fp64 oracle with the per-element bound of
oracle/bounds.py; the epilogue statistics and the norm-backward sums per (n, c)."""
import collections
import ctypes as C
import zlib

import pytest
import torch

from mra_gan_b200 import _lib, ops
from mra_gan_b200.ops import ConvGeom
from oracle import bounds as B
from oracle import ops_ref as R

G = ConvGeom
# kernel: the route expected for the three ops -- "gather" (gather / halo kernels + wgrad_tc_kernel), "stem", "head",
# "im2col", "convT1" (the lowerings of conv_special.cuh) or "fp32" (CUDA-core kernels, channel counts of any size)
# shared: wgrad work items split between CTAs (wgrad_fixup_kernel runs) -- True / False, None where not asserted
# cc: ops (0 fprop, 1 dgrad) of a "gather" case that stay on the CUDA cores: the strided dgrad form with k < stride
Case = collections.namedtuple("Case", "kernel g dims n shared pair_min0 cc", defaults=(None, False, ()))
LOWERING = {"gather": 0, "stem": 1, "head": 2, "convT1": 2, "im2col": 3, "fp32": 0}

CASES = [
    # -- gather / halo kernels: channel pairs (reduction side -> output side), k, stride, padding
    Case("gather", G(64, 64, 3, 1, 1), (9, 7, 5), 1),
    Case("gather", G(192, 320, 3, 1, 0), (5, 5, 6), 2),            # 5 n tiles of 64 (fprop), 3 (dgrad); Km 320
    Case("gather", G(384, 64, 3, 2, 1), (9, 8, 7), 3),             # odd extents, batch 3
    Case("gather", G(128, 192, 4, 2, 2), (7, 7, 7), 2),            # k4 pad 2, Km 192: ragged second m tile
    Case("gather", G(256, 384, 2, 2, 0), (8, 6, 10), 1),           # k2
    Case("gather", G(320, 192, 2, 1, 1), (6, 5, 7), 2),            # k2 pad 1
    Case("gather", G(64, 128, 1, 1, 0), (5, 7, 11), 5),            # k1, batch 5
    Case("gather", G(64, 64, 1, 2, 0), (9, 9, 9), 2, cc=(1,)),     # k1 stride 2 (dgrad: phases without a tap)
    Case("gather", G(512, 64, 3, 1, 2), (3, 3, 3), 1),             # pad 2 > output of the unpadded conv
    Case("gather", G(64, 512, 3, 1, 0), (4, 5, 3), 2),
    Case("gather", G(128, 128, 3, 1, 1), (1, 6, 9), 2),            # an axis of extent 1
    Case("gather", G(64, 64, 3, 1, 1), (3, 3, 150), 1),            # w longer than one box
    Case("gather", G(128, 64, 3, 1, 0), (13, 11, 7), 1),           # prime extents
    Case("gather", G(64, 64, 3, 1, 1), (17, 13, 11), 2),           # uneven tile count over the persistent grid
    Case("gather", G(192, 128, 4, 1, 3), (3, 4, 5), 3),            # k4 pad 3
    Case("gather", G(64, 256, 4, 2, 0), (9, 10, 11), 1),           # k4 stride 2 pad 0
    Case("gather", G(256, 64, 4, 2, 3), (5, 6, 4), 2),             # k4 stride 2 pad 3
    Case("gather", G(64, 128, 3, 2, 0), (7, 8, 9), 5),
    Case("gather", G(128, 64, 2, 2, 1), (5, 7, 6), 3),             # k2 stride 2 pad 1
    # -- ConvTranspose3d, output_padding 0 and 1
    Case("gather", G(192, 64, 3, 2, 1, True, 1), (5, 4, 6), 2),
    Case("gather", G(64, 320, 4, 2, 1, True, 0), (3, 4, 5), 1),
    Case("gather", G(128, 128, 2, 2, 0, True, 0), (4, 5, 3), 3),
    Case("gather", G(64, 64, 3, 2, 0, True, 1), (4, 3, 5), 2),
    Case("gather", G(256, 128, 4, 2, 3, True, 1), (4, 5, 6), 1),
    Case("gather", G(64, 64, 1, 2, 0, True, 1), (4, 3, 5), 2, cc=(0,)),
    Case("gather", G(128, 64, 3, 1, 1, True, 0), (5, 6, 7), 2),    # stride 1
    Case("gather", G(384, 192, 2, 2, 1, True, 1), (3, 3, 4), 5),
    # -- wgrad: items shared between CTAs or not, CTA pairs, Km 192, transposed with shared items
    Case("gather", G(64, 128, 3, 2, 1), (32, 32, 32), 1, shared=True),
    Case("gather", G(64, 192, 3, 1, 1), (12, 12, 12), 2, shared=True),          # Km 192
    Case("gather", G(128, 64, 3, 2, 1, True, 1), (12, 12, 12), 2, shared=True),
    Case("gather", G(512, 64, 3, 1, 1), (4, 4, 4), 1, shared=False),
    Case("gather", G(256, 256, 3, 1, 1), (6, 5, 4), 2, pair_min0=True),         # CTA pairs, Km 256
    Case("gather", G(256, 512, 3, 1, 1), (3, 4, 3), 1, pair_min0=True),         # CTA pairs, Km 512
    # -- stem: Cin = 1
    Case("stem", G(1, 64, 2, 1, 0), (6, 7, 9), 2),
    Case("stem", G(1, 128, 3, 1, 0), (5, 9, 11), 3),
    Case("stem", G(1, 192, 5, 1, 0), (7, 8, 9), 1),
    Case("stem", G(1, 64, 7, 1, 0), (9, 10, 12), 2),
    Case("stem", G(1, 128, 8, 1, 0), (9, 9, 10), 1),
    # -- head: Cout = 1
    Case("head", G(64, 1, 2, 1, 0), (5, 6, 7), 2),
    Case("head", G(128, 1, 4, 1, 1), (6, 7, 5), 1),
    Case("head", G(192, 1, 7, 1, 6), (4, 5, 6), 2),
    Case("head", G(64, 1, 8, 1, 0), (9, 9, 10), 1),
    Case("head", G(64, 1, 4, 1, 3), (5, 4, 6), 3),
    Case("head", G(320, 1, 2, 1, 1), (4, 5, 3), 2),
    # -- im2col: Cin = 1, stride 2, or stride 1 with padding
    Case("im2col", G(1, 64, 4, 2, 1), (9, 10, 8), 2),
    Case("im2col", G(1, 128, 3, 2, 0), (9, 7, 8), 1),
    Case("im2col", G(1, 64, 3, 1, 1), (6, 7, 5), 2),
    Case("im2col", G(1, 192, 4, 1, 2), (5, 6, 4), 1),
    Case("im2col", G(1, 64, 1, 2, 0), (7, 6, 9), 3),
    # -- ConvTranspose3d(C -> 1): the mirror of the im2col lowering
    Case("convT1", G(128, 1, 4, 2, 1, True, 0), (5, 6, 4), 2),
    Case("convT1", G(64, 1, 3, 2, 1, True, 1), (5, 6, 7), 1),
    Case("convT1", G(192, 1, 2, 2, 0, True, 0), (4, 4, 5), 2),
    # -- stem and head with lines up to 256 wide (the Z line of shift_sum: the stem's output width, the head's input)
    Case("stem", G(1, 64, 2, 1, 0), (3, 3, 187), 1),               # Z line 186
    Case("stem", G(1, 64, 2, 1, 0), (3, 3, 188), 1),               # 187
    Case("stem", G(1, 128, 2, 1, 0), (3, 3, 199), 1),              # 198
    Case("stem", G(1, 64, 2, 1, 0), (3, 3, 256), 2),               # 255
    Case("head", G(64, 1, 7, 1, 0), (7, 7, 186), 1),
    Case("head", G(64, 1, 7, 1, 0), (7, 7, 187), 1),
    Case("head", G(64, 1, 7, 1, 3), (7, 7, 198), 1),               # the resnet head on a 192-wide patch
    Case("head", G(128, 1, 4, 1, 1), (4, 4, 256), 2),
    # -- fp32: CUDA-core kernels, channel counts that are not multiples of 8 (scalar loads)
    Case("fp32", G(12, 20, 3, 1, 1), (5, 6, 7), 2),
    Case("fp32", G(5, 3, 4, 2, 1), (8, 7, 6), 1),
    Case("fp32", G(7, 9, 3, 2, 1, True, 1), (4, 5, 3), 2),
    Case("fp32", G(1, 13, 2, 1, 0), (6, 5, 7), 3),
    Case("fp32", G(11, 1, 4, 1, 3), (5, 4, 6), 2),
    Case("fp32", G(64, 64, 3, 1, 1), (9, 7, 5), 1),
    Case("fp32", G(192, 64, 2, 2, 0), (6, 5, 7), 2),
]


def cid(c):
    g = c.g
    return "%s_c%d-%d_k%d_s%d_p%d%s_%s_n%d" % (c.kernel, g.cin, g.cout, g.k, g.stride, g.pad,
                                             ("T%d" % g.output_padding) if g.transposed else "",
                                             "x".join(map(str, c.dims)), c.n)


def desc(c):
    """host-side descriptor of a case (the dispatcher's view)"""
    d = _lib.ConvDesc()
    g = c.g
    d.n, d.cin, d.cout = c.n, g.cin, g.cout
    d.din, d.hin, d.win = c.dims
    d.dout, d.hout, d.wout = g.out_dims(c.dims)
    d.k, d.stride, d.pad, d.transposed = g.k, g.stride, g.pad, int(g.transposed)
    d.dtype = _lib.MRA_F32 if c.kernel == "fp32" else _lib.MRA_BF16
    return d


def route(c, which):
    """kernel family of op ``which`` for the report: the lowering, else halo / gather / wgrad, or cuda-core"""
    if c.kernel == "fp32" or which in c.cc:
        return "cuda-core"
    if c.kernel != "gather":
        return c.kernel
    if which == 2:
        return "wgrad"
    words = ops.schedule_describe(c.g, c.n, c.dims, which)
    return "halo" if words[1] > 0 else "gather"


def wgrad_schedule(c):
    """(CTA pairs?, any work item split between stream-K units?) of the wgrad launch, from the host walk of its
    schedule (mra_debug_schedule, layout in include/mra_gan_b200.h)"""
    w = ops.schedule_describe(c.g, c.n, c.dims, 2)
    pair, n_groups, kblocks = w[1], w[4], w[6]
    at = 10 + 5 * n_groups
    segs = [w[at + 1 + 9 * i: at + 10 + 9 * i] for i in range(w[at])]
    assert segs, "empty wgrad schedule"
    return bool(pair), any(s[7] > 0 or s[8] < kblocks for s in segs)


WORST = collections.defaultdict(float)


@pytest.fixture(scope="module")
def report():
    yield WORST
    for k in sorted(WORST):
        print("worst error / bound  %-22s %.3f" % (k, WORST[k]))


def _note(key, ratio):
    WORST[key] = max(WORST[key], ratio)


def _operands(c, dtype):
    g = c.g
    gen = torch.Generator().manual_seed(zlib.crc32(cid(c).encode()))
    x = torch.randn((c.n,) + c.dims + (g.cin,), generator=gen).to(dtype)
    w = (torch.randn((g.taps, g.cout, g.cin), generator=gen) / (g.taps * g.cin) ** 0.5).to(dtype)
    b = torch.randn((g.cout,), generator=gen)
    dy = torch.randn((c.n,) + g.out_dims(c.dims) + (g.cout,), generator=gen).to(dtype)
    xh = torch.randn((c.n,) + c.dims + (g.cin,), generator=gen)
    return x, w, b, dy, xh


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=cid)
def test_conv_envelope(c, report, monkeypatch):
    g, dims, n = c.g, c.dims, c.n
    dtype = torch.float32 if c.kernel == "fp32" else torch.bfloat16
    tcore = c.kernel != "fp32"
    I = ops.impl()
    d = desc(c)
    on_tc = [tcore and which not in c.cc for which in range(3)]
    for which in range(3):
        assert I.conv_uses_tensor_cores(g, n, dims, dtype, which) == on_tc[which], which
    low = int(I.L.mra_conv3d_lowering(C.byref(d)))
    assert low == LOWERING[c.kernel]
    if c.pair_min0:
        monkeypatch.setenv("MRA_WGRAD_PAIR_MIN", "0")
    if c.kernel == "gather":
        pair, shared = wgrad_schedule(c)
        assert pair or not c.pair_min0, "CTA pairs expected"
        assert c.shared is None or shared == c.shared, "wgrad items shared between CTAs: %s" % shared
    acc = [B.acc_type(dtype, on_tc[which], low, which) for which in range(3)]
    fam = [route(c, which) + "-" + ("fprop", "dgrad", "wgrad")[which] for which in range(3)]

    x, w, b, dy, xh = _operands(c, dtype)
    xd, wd, bd, dyd = x.cuda(), w.cuda(), b.cuda(), dy.cuda()

    # fprop + bias, every activation; epilogue statistics of the pre-activation output
    pre, mag = B.fprop_ref(x, w, b, g)
    for act in (R.ACT_NONE, R.ACT_LRELU, R.ACT_TANH, R.ACT_SIGMOID):
        y, st = I.conv_fprop(xd, wd, bd, g, act=act, slope=0.2, want_stats=act == R.ACT_NONE)
        assert I.tc_error() == 0
        r = B.check_output(y, pre, mag, acc[0], act, 0.2, "fprop act %d" % act)
        if st is not None:
            r = max(r, B.check_stats(st, pre, mag, dtype, acc[0], "fprop statistics"))
        _note(fam[0], r)
    del pre, mag

    # dgrad, and the norm-backward statistics fused into it where the kernel supports them
    wT = I.pack_weight_t(wd, dtype)
    dx = I.conv_dgrad(dyd, wT, g, dims)
    assert I.tc_error() == 0
    ref, mag = B.dgrad_ref(dy, w.transpose(1, 2).contiguous(), g, dims)
    _note(fam[1], B.check_output(dx, ref, mag, acc[1], what="dgrad"))
    if tcore and I.conv_dgrad_nstats_supported(g, n, dims, dtype):
        act, slope = (R.ACT_RELU, 0.0) if n % 2 else (R.ACT_LRELU, 0.2)
        ns = 0.0 if act == R.ACT_RELU else slope
        ya = torch.where(xh > 0, xh, xh * ns).to(dtype)
        dx2, sums = I.conv_dgrad_nstats(dyd, wT, g, dims, ya.cuda(), act, slope)
        assert I.tc_error() == 0
        if I.L.mra_conv3d_workspace_size(C.byref(d), 1) == 0:
            assert torch.equal(dx2, dx), "dgrad_nstats: dx differs from the plain dgrad"
        else:                    # the plain dgrad took the split-K path: the same sums in another order
            B.check_output(dx2, ref, mag, acc[1], what="dgrad_nstats dx")
        _, bound = B.output_bound(ref, mag, dtype, acc[1])
        y64 = ya.double()
        wgt = torch.where(y64 > 0, torch.ones_like(y64), torch.full_like(y64, ns))
        for j, f in enumerate((wgt, y64)):
            _note(fam[1] + "-nstats", B.check_elements(sums[..., j], (ref * f).sum((1, 2, 3)),
                                                        (bound * f.abs()).sum((1, 2, 3)), "nstats %d" % j, ("n", "c")))
    del ref, mag

    # wgrad + dbias, fresh and added into nonzero buffers
    dw, db = I.conv_wgrad(xd, dyd, g, want_bias=True)
    assert I.tc_error() == 0
    ref, mag = B.wgrad_ref(x, dy, g)
    _note(fam[2], B.check_elements(dw, ref, B.CU[acc[2]] * mag, "wgrad", B.W_NAMES))
    _note("dbias", B.check_dbias(db, dy))
    base_w, base_b = torch.randn_like(dw), torch.randn_like(db)
    aw, ab = base_w.clone(), base_b.clone()
    I.conv_wgrad(xd, dyd, g, want_bias=True, acc_dw=aw, acc_db=ab)
    assert I.tc_error() == 0
    bw = base_w.cpu().double()
    _note(fam[2], B.check_elements(aw, ref + bw, B.CU[acc[2]] * mag + 2.0 ** -23 * bw.abs(), "wgrad accumulate",
                                   B.W_NAMES))
    _note("dbias", B.check_dbias(ab, dy, "dbias accumulate", base_b))

    # the lowerings' shared workspace: the expanded operand written by one call is reused by the next, same bits
    if low:
        _, ws = I.conv_shared_workspace(g, n, dims, dtype, "cuda")
        if low in (1, 3):
            I.conv_fprop(xd, wd, bd, g, ws=ws)
            dw_r, _ = I.conv_wgrad(xd, dyd, g, ws=ws, reuse=True)
            assert torch.equal(dw_r, dw), "wgrad after fprop with the workspace reused"
        else:
            I.conv_wgrad(xd, dyd, g, ws=ws)
            dx_r = I.conv_dgrad(dyd, wT, g, dims, ws=ws, reuse=True)
            assert torch.equal(dx_r, dx), "dgrad after wgrad with the workspace reused"
        assert I.tc_error() == 0
