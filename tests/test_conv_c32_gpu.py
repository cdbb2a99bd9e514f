"""Convolutions whose channel counts are multiples of 32 but not of 64 (32, 96, 160) on the tensor cores: K chunks
zero-filled by TMA past the channel extent, the last 64-wide N tile masked in the epilogue and the wgrad flush.  Every
case runs the element-by-element checks of test_conv_envelope_gpu (fp64 oracle, per-element bounds of
oracle/bounds.py): fprop with every activation and its statistics, dgrad, dgrad_nstats, wgrad + dbias fresh and
accumulated, workspace reuse of the lowerings.  On top: the stride-2 transposed layer of the ngf = 32 generator under
the gather switches, bit-reproducible shared wgrad items, and guard words around every output buffer (the masked
columns are where a stray store would land)."""
import ctypes as C

import pytest
import torch

import test_conv_envelope_gpu as EV
from mra_gan_b200 import _lib, ops
from mra_gan_b200.ops import ConvGeom as G
from oracle import ops_ref as R

Case = EV.Case

CASES = [
    # -- per-tap gather kernel + wgrad_tc_kernel: 32 / 96 / 160 on either side and on both
    Case("gather", G(32, 32, 3, 1, 1), (9, 7, 5), 1),
    Case("gather", G(32, 64, 3, 2, 1), (9, 8, 7), 2),             # G.d1 / D.1 at ngf = ndf = 32 (k3 s2)
    Case("gather", G(32, 64, 4, 2, 1), (8, 9, 10), 3),            # D.1 (k4 s2)
    Case("gather", G(64, 32, 3, 1, 0), (13, 11, 7), 1),           # prime extents
    Case("gather", G(96, 160, 2, 1, 1), (6, 5, 7), 2),            # 3 N tiles of 64, the last one masked
    Case("gather", G(160, 96, 3, 2, 0), (7, 8, 9), 5),
    Case("gather", G(32, 256, 1, 1, 0), (5, 7, 11), 5),           # k1
    Case("gather", G(256, 32, 4, 2, 3), (5, 6, 4), 2),
    Case("gather", G(32, 32, 1, 2, 0), (9, 9, 9), 2, cc=(1,)),    # k1 stride 2: dgrad phases without a tap
    Case("gather", G(96, 32, 2, 2, 1), (5, 7, 6), 3),
    Case("gather", G(32, 96, 3, 1, 1), (3, 3, 150), 1),           # w longer than one box
    # -- ConvTranspose3d, output_padding 0 and 1
    Case("gather", G(64, 32, 3, 2, 1, True, 1), (4, 5, 6), 2),    # G.u2 at ngf = 32
    Case("gather", G(32, 96, 4, 2, 1, True, 0), (3, 4, 5), 1),
    Case("gather", G(160, 32, 2, 2, 0, True, 0), (4, 5, 3), 3),
    Case("gather", G(32, 32, 3, 1, 1, True, 0), (5, 6, 7), 2),    # stride 1
    Case("gather", G(32, 64, 1, 2, 0, True, 1), (4, 3, 5), 2, cc=(0,)),
    # -- wgrad items shared between CTAs (fix-up kernel), 32 channels on the shifted / dense side
    Case("gather", G(32, 64, 3, 2, 1), (32, 32, 32), 1, shared=True),
    Case("gather", G(64, 32, 3, 1, 1), (12, 12, 12), 2, shared=True),
    Case("gather", G(64, 32, 3, 2, 1, True, 1), (12, 12, 12), 2, shared=True),
    # -- the channel-expanded lowerings
    Case("stem", G(1, 32, 7, 1, 0), (9, 10, 12), 2),              # G stem at ngf = 32
    Case("stem", G(1, 96, 2, 1, 0), (6, 7, 9), 1),
    Case("stem", G(1, 32, 2, 1, 0), (3, 3, 187), 1),              # Z line 186
    Case("stem", G(1, 32, 2, 1, 0), (3, 3, 256), 2),
    Case("head", G(32, 1, 7, 1, 3), (7, 7, 9), 2),                # G head at ngf = 32
    Case("head", G(96, 1, 2, 1, 0), (5, 6, 7), 1),
    Case("head", G(32, 1, 7, 1, 0), (7, 7, 187), 1),
    Case("im2col", G(1, 32, 4, 2, 1), (9, 10, 8), 2),             # D.0 at ndf = 32
    Case("im2col", G(1, 32, 1, 2, 0), (7, 6, 9), 3),              # the pixel discriminator's first layer, strided
    Case("im2col", G(1, 96, 3, 1, 1), (6, 7, 5), 2),
    Case("convT1", G(32, 1, 4, 2, 1, True, 0), (5, 6, 4), 2),
    Case("convT1", G(96, 1, 3, 2, 1, True, 1), (5, 6, 7), 1),
]

U2 = Case("gather", G(64, 32, 3, 2, 1, True, 1), (6, 5, 7), 2)


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=EV.cid)
def test_conv_c32(c, monkeypatch):
    EV.test_conv_envelope(c, EV.WORST, monkeypatch)
    assert ops.impl().tc_error() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("env", ["MRA_GATHER_NOPAIR", "MRA_GATHER_NOMERGE", "MRA_GATHER_PHASE"])
def test_u2_c32_under_gather_switches(env, monkeypatch):
    """the merged parity phases of the transposed layer at cn = 32, without phase pairs, as 8 launches, and with the
    opt-in phase-halo kernel asked for (it declines 32-channel shapes; the per-tap kernel takes the launch)"""
    monkeypatch.setenv(env, "1")
    EV.test_conv_envelope(U2, EV.WORST, monkeypatch)
    assert ops.impl().tc_error() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("c", [CASES[16], CASES[17], CASES[18]], ids=EV.cid)
def test_c32_shared_wgrad_is_reproducible(c):
    """work items split between CTAs are added in K order by the fix-up kernel: the same bits every run"""
    I = ops.impl()
    x, w, b, dy, xh = EV._operands(c, torch.bfloat16)
    xd, dyd = x.cuda(), dy.cuda()
    assert EV.wgrad_schedule(c)[1], "expected work items shared between CTAs"
    runs = [I.conv_wgrad(xd, dyd, c.g, want_bias=True) for _ in range(3)]
    assert I.tc_error() == 0
    for dw, db in runs[1:]:
        assert torch.equal(dw, runs[0][0]) and torch.equal(db, runs[0][1])


GUARD_CASES = [
    Case("gather", G(64, 32, 3, 1, 1), (7, 6, 9), 2),             # cn = 32 fprop, ck = 32 dgrad, Kn = 64 / Km = 32 wgrad
    Case("gather", G(96, 160, 3, 2, 1), (7, 6, 5), 2),            # masked last N tile (fprop 160, dgrad 96)
    Case("gather", G(64, 32, 3, 2, 1, True, 1), (5, 6, 7), 2),    # merged phases, ConvTranspose3d wgrad (n_stride != 1)
    Case("gather", G(32, 64, 3, 2, 1), (32, 32, 32), 1, shared=True),   # shared items: fix-up kernel at Kn = 32
    Case("stem", G(1, 32, 7, 1, 0), (9, 10, 12), 2),
    Case("head", G(32, 1, 7, 1, 3), (7, 7, 9), 2),
    Case("im2col", G(1, 96, 4, 2, 1), (9, 10, 8), 2),
    Case("convT1", G(32, 1, 4, 2, 1, True, 0), (5, 6, 4), 2),
]
GUARD = 4096          # elements on either side


def _guarded(shape, dtype):
    """(view, buffer): a contiguous view into a buffer padded with -0.0 on both sides"""
    n = 1
    for s in shape:
        n *= s
    buf = torch.full((GUARD + n + GUARD,), -0.0, dtype=dtype, device="cuda")
    return buf[GUARD:GUARD + n].view(shape), buf


def _intact(buf, what):
    bits = {torch.bfloat16: torch.int16, torch.float32: torch.int32, torch.float64: torch.int64}[buf.dtype]
    neg0 = torch.tensor([-0.0], dtype=buf.dtype).view(bits).item()
    b = buf.view(bits).cpu()
    assert bool((b[:GUARD] == neg0).all()), what + ": a store landed BEFORE the buffer"
    assert bool((b[-GUARD:] == neg0).all()), what + ": a store landed PAST the buffer"


@pytest.mark.gpu
@pytest.mark.parametrize("c", GUARD_CASES, ids=EV.cid)
def test_c32_outputs_stay_inside_their_buffers(c):
    I = ops.impl()
    g, n, dims = c.g, c.n, c.dims
    out_dims = g.out_dims(dims)
    x, w, b, dy, xh = EV._operands(c, torch.bfloat16)
    xd, wd, bd, dyd = x.cuda(), w.cuda(), b.cuda(), dy.cuda()
    wT = I.pack_weight_t(wd, torch.bfloat16)
    st = I._stream()
    p = lambda t: C.c_void_p(t.data_ptr() if t is not None else 0)
    ref_y, ref_stats = I.conv_fprop(xd, wd, bd, g, want_stats=c.kernel not in ("head", "convT1"))
    ref_dx = I.conv_dgrad(dyd, wT, g, dims)
    ref_dw, ref_db = I.conv_wgrad(xd, dyd, g, want_bias=True)

    def ws(which):
        d = I._conv_desc(g, n, dims, out_dims, _lib.MRA_BF16)
        nb = int(I.L.mra_conv3d_workspace_size(C.byref(d), which))
        return d, (torch.empty(nb, dtype=torch.uint8, device="cuda") if nb else None), nb

    # fprop: y and the statistics
    y, ybuf = _guarded((n,) + out_dims + (g.cout,), torch.bfloat16)
    stats, sbuf = (_guarded((n, g.cout, 2), torch.float64) if ref_stats is not None else (None, None))
    d, wsp, nb = ws(0)
    _lib.check(I.L.mra_conv3d_fprop(C.byref(d), p(xd), p(wd), p(bd), p(y), p(stats), p(wsp), nb, st), "fprop")
    torch.cuda.synchronize()
    _intact(ybuf, "fprop y")
    assert torch.equal(y, ref_y)
    if stats is not None:
        _intact(sbuf, "fprop statistics")
        assert torch.allclose(stats, ref_stats, rtol=1e-9, atol=1e-9)
    # dgrad, and the norm-backward sums where supported
    dx, xbuf = _guarded((n,) + dims + (g.cin,), torch.bfloat16)
    d, wsp, nb = ws(1)
    _lib.check(I.L.mra_conv3d_dgrad(C.byref(d), p(dyd), p(wT), p(dx), p(wsp), nb, st), "dgrad")
    torch.cuda.synchronize()
    _intact(xbuf, "dgrad dx")
    assert torch.equal(dx, ref_dx)
    if I.conv_dgrad_nstats_supported(g, n, dims, torch.bfloat16):
        ya = torch.where(xh > 0, xh, xh * 0.2).to(torch.bfloat16).cuda()
        dx2, xbuf2 = _guarded((n,) + dims + (g.cin,), torch.bfloat16)
        sums, ubuf = _guarded((n, g.cin, 2), torch.float64)
        _lib.check(I.L.mra_conv3d_dgrad_nstats(C.byref(d), p(dyd), p(wT), p(dx2), p(ya), R.ACT_LRELU, C.c_float(0.2), p(sums), p(wsp), nb, st), "dgrad_nstats")
        torch.cuda.synchronize()
        _intact(xbuf2, "dgrad_nstats dx")
        _intact(ubuf, "dgrad_nstats sums")
    # wgrad + dbias
    dw, wbuf = _guarded((g.taps, g.cout, g.cin), torch.float32)
    db, bbuf = _guarded((g.cout,), torch.float32)
    d, wsp, nb = ws(2)
    _lib.check(I.L.mra_conv3d_wgrad(C.byref(d), p(xd), p(dyd), p(dw), p(db), p(wsp), nb, st), "wgrad")
    torch.cuda.synchronize()
    _intact(wbuf, "wgrad dw")
    _intact(bbuf, "wgrad db")
    assert torch.allclose(dw, ref_dw, rtol=1e-5, atol=1e-6) and torch.allclose(db, ref_db, rtol=1e-5, atol=1e-6)
    assert I.tc_error() == 0
