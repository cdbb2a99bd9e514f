"""The per-element conv checker (oracle/bounds.py) pinned on the CPU: it accepts the arithmetic of the kernels (fp32
accumulation of the operands as stored, output rounded to bf16), and it rejects local mutations that the global
rel-L2 < 1e-2 check of a whole tensor lets pass."""
import pytest
import torch

from mra_gan_b200.ops import ConvGeom
from oracle import bounds as B
from oracle import ops_ref as R
from oracle.functional import rel_l2

F32 = R.RefImpl(torch.float32)


def _case(g, dims, n, seed=0, dtype=torch.bfloat16):
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn((n,) + dims + (g.cin,), generator=gen).to(dtype)
    w = (torch.randn((g.taps, g.cout, g.cin), generator=gen) / (g.taps * g.cin) ** 0.5).to(dtype)
    b = torch.randn((g.cout,), generator=gen)
    dy = torch.randn((n,) + g.out_dims(dims) + (g.cout,), generator=gen).to(dtype)
    return x, w, b, dy


ACCEPT = [
    (ConvGeom(16, 24, 3, 1, 0), (7, 6, 9), 2),
    (ConvGeom(16, 8, 3, 2, 1), (9, 8, 7), 2),
    (ConvGeom(8, 16, 4, 2, 1), (8, 10, 6), 1),
    (ConvGeom(8, 8, 4, 1, 1), (5, 6, 7), 2),
    (ConvGeom(16, 8, 3, 2, 1, True, 1), (4, 5, 3), 2),
    (ConvGeom(8, 16, 4, 2, 1, True, 0), (3, 4, 5), 1),
    (ConvGeom(1, 16, 7, 1, 0), (9, 8, 10), 1),
    (ConvGeom(16, 1, 4, 1, 0), (7, 6, 8), 2),
]


def _gid(c):
    g, dims, n = c
    return "c%d-%d_k%d_s%d_p%d_%s" % (g.cin, g.cout, g.k, g.stride, g.pad, "T" if g.transposed else "C")


@pytest.mark.parametrize("case", ACCEPT, ids=_gid)
def test_checker_accepts_fp32_accumulation_with_bf16_outputs(case):
    """What a kernel computes: the bf16 operands multiplied and summed in fp32 (here by the CPU), the output rounded to
    bf16 once; fused activations, epilogue statistics of the fp32 sums, dw in fp32, dbias summed in fp32."""
    g, dims, n = case
    x, w, b, dy = _case(g, dims, n)
    xf, wf, dyf = x.float(), w.float(), dy.float()
    for act, slope in ((R.ACT_NONE, 0.2), (R.ACT_LRELU, 0.2), (R.ACT_TANH, 0.2), (R.ACT_SIGMOID, 0.2)):
        y, st = F32.conv_fprop(xf, wf, b, g, act=act, slope=slope, want_stats=act == R.ACT_NONE)
        assert B.check_fprop(y.to(torch.bfloat16), x, w, b, g, "tc", act, slope, got_stats=st) <= 1
    dx = F32.conv_dgrad(dyf, wf.transpose(1, 2).contiguous(), g, dims).to(torch.bfloat16)
    assert B.check_dgrad(dx, dy, w.transpose(1, 2).contiguous(), g, "tc") <= 1
    dw, db = F32.conv_wgrad(xf, dyf, g, want_bias=True)
    assert B.check_wgrad(dw, x, dy, g, "tc", got_db=db) <= 1
    base_w, base_b = torch.randn_like(dw), torch.randn_like(db)
    assert B.check_wgrad(base_w + dw, x, dy, g, "tc", got_db=base_b + db, base_dw=base_w, base_db=base_b) <= 1
    # fp32 storage: the CUDA-core constant, no output rounding
    y, st = F32.conv_fprop(xf, wf, b, g, want_stats=True)
    assert B.check_fprop(y, xf, wf, b, g, "fma", got_stats=st) <= 1


def test_acc_type_follows_the_route():
    assert B.acc_type(torch.float32, False) == "fma"
    assert B.acc_type(torch.bfloat16, True) == "tc"
    assert [B.acc_type(torch.bfloat16, True, 1, w) for w in range(3)] == ["tc", "tc_bf16", "tc"]       # stem: Z in dgrad
    assert [B.acc_type(torch.bfloat16, True, 2, w) for w in range(3)] == ["tc_bf16", "tc", "tc"]       # head: Z in fprop
    assert [B.acc_type(torch.bfloat16, True, 3, w) for w in range(3)] == ["tc", "tc_bf16", "tc"]       # im2col: dE in dgrad


# ----------------------------------------------------------------------------------------------------------------------
# mutations that pass the global rel-L2 < 1e-2 and must not pass the checker
# ----------------------------------------------------------------------------------------------------------------------
def _fprop_bf16(x, w, b, g):
    y, st = F32.conv_fprop(x.float(), w.float(), b, g, want_stats=True)
    return y.to(torch.bfloat16), st


def _rejected(check):
    with pytest.raises(B.BoundError):
        check()


def test_rejects_one_zeroed_output_element():
    g, dims, n = ConvGeom(64, 64, 3, 1, 0), (10, 10, 10), 2
    x, w, b, _ = _case(g, dims, n, seed=1)
    y, _ = _fprop_bf16(x, w, b, g)
    ym = y.clone()
    ym[1, 3, 4, 5, 17] = 0
    y_ref, _ = R.RefImpl(torch.float64).conv_fprop(x.double(), w.double(), b.double(), g)
    assert rel_l2(ym, y_ref) < 1e-2
    assert B.check_fprop(y, x, w, b, g, "tc") <= 1
    _rejected(lambda: B.check_fprop(ym, x, w, b, g, "tc"))


def test_rejects_a_tap_dropped_on_the_last_w_column():
    """the ragged edge of a gather / halo tile: the centre tap missing from the outputs of the last w column only"""
    g, dims, n = ConvGeom(16, 32, 3, 1, 0), (4, 4, 242), 1
    x, w, b, _ = _case(g, dims, n, seed=2)
    y, _ = _fprop_bf16(x, w, b, g)
    w0 = w.clone()
    w0[13] = 0
    y0, _ = _fprop_bf16(x, w0, b, g)
    ym = y.clone()
    ym[:, :, :, -1] = y0[:, :, :, -1]
    y_ref, _ = R.RefImpl(torch.float64).conv_fprop(x.double(), w.double(), b.double(), g)
    assert rel_l2(ym, y_ref) < 1e-2
    _rejected(lambda: B.check_fprop(ym, x, w, b, g, "tc"))


def test_rejects_a_k_chunk_lost_on_one_tile():
    """channels 64..127 of one tap missing on one tile of 128 consecutive output positions"""
    g, dims, n = ConvGeom(128, 16, 3, 1, 0), (22, 22, 22), 2
    x, w, b, _ = _case(g, dims, n, seed=3)
    y, _ = _fprop_bf16(x, w, b, g)
    w0 = w.clone()
    w0[4, :, 64:128] = 0
    y0, _ = _fprop_bf16(x, w0, b, g)
    flat, flat0 = y.clone().view(-1, g.cout), y0.view(-1, g.cout)
    flat[5 * 128:6 * 128] = flat0[5 * 128:6 * 128]
    ym = flat.view(y.shape)
    y_ref, _ = R.RefImpl(torch.float64).conv_fprop(x.double(), w.double(), b.double(), g)
    assert rel_l2(ym, y_ref) < 1e-2
    _rejected(lambda: B.check_fprop(ym, x, w, b, g, "tc"))


def test_rejects_a_tile_counted_twice_in_one_channel_sum():
    g, dims, n = ConvGeom(16, 64, 3, 1, 0), (14, 14, 14), 2
    x, w, b, _ = _case(g, dims, n, seed=4)
    y, st = _fprop_bf16(x, w, b, g)
    pre, _ = B.fprop_ref(x, w, b, g)
    tile = pre[1].reshape(-1, g.cout)[2 * 128:3 * 128].sum(0)      # one 128-position tile of sample 1, every channel
    c = 37
    stm = st.clone()
    stm[1, c, 0] += tile[c]
    _, st_ref = R.RefImpl(torch.float64).conv_fprop(x.double(), w.double(), b.double(), g, want_stats=True)
    assert rel_l2(stm, st_ref) < 1e-2
    assert B.check_fprop(y, x, w, b, g, "tc", got_stats=st) <= 1
    _rejected(lambda: B.check_fprop(y, x, w, b, g, "tc", got_stats=stm))


def test_rejects_a_k_block_missing_from_dw():
    """the contribution of one 128-position K block to one tap of dw missing"""
    g, dims, n = ConvGeom(16, 16, 4, 1, 1), (24, 24, 24), 2
    x, _, _, dy = _case(g, dims, n, seed=5)
    dw, _ = F32.conv_wgrad(x.float(), dy.float(), g)
    blk = torch.zeros_like(dy)
    blk.view(-1, g.cout)[7 * 128:8 * 128] = dy.view(-1, g.cout)[7 * 128:8 * 128]
    part, _ = F32.conv_wgrad(x.float(), blk.float(), g)
    dwm = dw.clone()
    dwm[21] -= part[21]
    dw_ref, _ = R.RefImpl(torch.float64).conv_wgrad(x.double(), dy.double(), g)
    assert rel_l2(dwm, dw_ref) < 1e-2
    assert B.check_wgrad(dw, x, dy, g, "tc") <= 1
    _rejected(lambda: B.check_wgrad(dwm, x, dy, g, "tc"))
