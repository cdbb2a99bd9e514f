"""GPU parity of every C-ABI op against the op-level oracle (oracle/ops_ref.py, torch CPU).
Tolerances (BASELINE.json north_star): rel-L2 <= 1e-4 on the fp32 path, <= 1e-2 on the bf16 path."""
import pytest
import torch

from mra_gan_b200 import ops
from mra_gan_b200.ops import ConvGeom
from oracle import bounds as B
from oracle import ops_ref as R
from oracle.functional import rel_l2

pytestmark = pytest.mark.gpu
TOL = {torch.float32: 1e-4, torch.bfloat16: 1e-2}

CONVS = [
    # (geom, in_dims, N)
    (ConvGeom(1, 8, 7, 1, 0), (14, 14, 14), 2),            # stem-like (Cin=1)
    (ConvGeom(8, 1, 7, 1, 0), (14, 14, 14), 2),            # head-like (Cout=1)
    (ConvGeom(8, 16, 3, 2, 1), (12, 12, 12), 2),
    (ConvGeom(16, 16, 3, 1, 0), (10, 10, 10), 1),
    (ConvGeom(1, 8, 4, 2, 1), (12, 12, 12), 2),
    (ConvGeom(16, 24, 4, 1, 1), (7, 7, 7), 2),
    (ConvGeom(16, 8, 3, 2, 1, True, 1), (5, 6, 7), 2),
    (ConvGeom(16, 8, 4, 2, 1, True, 0), (4, 5, 3), 2),
]
TC_CONVS = [
    (ConvGeom(256, 256, 3, 1, 0), (10, 10, 10), 2),        # G.rb
    (ConvGeom(64, 128, 3, 2, 1), (16, 16, 16), 1),         # G.d1
    (ConvGeom(64, 128, 4, 2, 1), (16, 16, 16), 2),         # D.2
    (ConvGeom(128, 512, 4, 1, 1), (10, 10, 10), 1),        # D.4-like, ragged 9^3 output
    (ConvGeom(256, 128, 3, 2, 1, True, 1), (6, 6, 6), 2),  # G.u1
    (ConvGeom(128, 64, 4, 2, 1, True, 0), (5, 5, 5), 1),   # UNet up
    (ConvGeom(64, 64, 3, 1, 1), (9, 7, 5), 1),             # zero-padded, odd dims
    (ConvGeom(1, 64, 7, 1, 0), (14, 15, 17), 2),           # G.c1 stem: channel-expanded lowering
    (ConvGeom(64, 1, 7, 1, 0), (14, 15, 17), 2),           # G.c4 head: channel-expanded lowering
    (ConvGeom(128, 1, 4, 1, 0), (7, 8, 9), 1),             # head-like, k4
    (ConvGeom(1, 64, 4, 2, 1), (12, 12, 12), 2),           # D.1: im2col lowering
    (ConvGeom(512, 1, 4, 1, 1), (7, 7, 7), 2),             # D.5: zero-padded head lowering
    (ConvGeom(128, 1, 4, 2, 1, True, 0), (6, 6, 6), 2),    # UNet outermost up-conv: mirror of the im2col lowering
    (ConvGeom(64, 1, 3, 2, 1, True, 1), (5, 6, 7), 1),     # ConvTranspose3d(C -> 1) with output padding
    (ConvGeom(128, 64, 3, 2, 1, True, 1), (12, 12, 12), 2),  # G.u2: 8 merged parity phases, several work items per CTA,
                                                             # deferred statistics across a sample boundary
    (ConvGeom(64, 128, 3, 2, 1), (15, 16, 17), 1),         # odd dims: the dgrad phases differ in extent -> unmerged launches
]


def gid(v):
    g, dims, n = v
    return "c%d-%d_k%d_s%d_p%d_%s_%s" % (g.cin, g.cout, g.k, g.stride, g.pad, "T" if g.transposed else "C",
                                         "x".join(map(str, dims)))


def _conv_case(g, dims, n, dtype, seed=0):
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn((n,) + dims + (g.cin,), generator=gen).to(dtype)
    w = (torch.randn((g.taps, g.cout, g.cin), generator=gen) / (g.taps * g.cin) ** 0.5).to(dtype)
    b = torch.randn((g.cout,), generator=gen)
    dy = torch.randn((n,) + g.out_dims(dims) + (g.cout,), generator=gen).to(dtype)
    return x, w, b, dy


def _acc(g, dims, n, dtype, which):
    """accumulation type of op ``which`` on the route the dispatcher picks (oracle/bounds.py)"""
    import ctypes as C
    I = ops.impl()
    tc = I.conv_uses_tensor_cores(g, n, dims, dtype, which)
    low = int(I.L.mra_conv3d_lowering(C.byref(I._conv_desc(g, n, dims, g.out_dims(dims), ops.MRA_BF16)))) if tc else 0
    return B.acc_type(dtype, tc, low, which)


def _check_conv(g, dims, n, dtype, expect_tc):
    """every element of fprop (+ bias, + LeakyReLU), dgrad, wgrad (+ dbias, fresh and accumulated) and every (n, c) of
    the epilogue statistics within the per-element bound of oracle/bounds.py"""
    I = ops.impl()
    x, w, b, dy = _conv_case(g, dims, n, dtype)
    dev = "cuda"
    xd, wd, bd, dyd = x.to(dev), w.to(dev), b.to(dev), dy.to(dev)
    for which in range(3):
        assert I.conv_uses_tensor_cores(g, n, dims, dtype, which) == expect_tc
    acc = [_acc(g, dims, n, dtype, which) for which in range(3)]
    # fprop (+bias, + epilogue statistics)
    y, st = I.conv_fprop(xd, wd, bd, g, want_stats=True)
    assert I.tc_error() == 0
    pre, mag = B.fprop_ref(x, w, b, g)
    B.check_output(y, pre, mag, acc[0], what="fprop")
    B.check_stats(st, pre, mag, dtype, acc[0], "epilogue stats")
    y2, _ = I.conv_fprop(xd, wd, None, g, act=ops.ACT_LRELU, slope=0.2)
    B.check_fprop(y2, x, w, None, g, acc[0], R.ACT_LRELU, 0.2, what="fprop+lrelu")
    # dgrad
    wT = I.pack_weight_t(wd, dtype)
    assert torch.equal(wT.cpu(), w.transpose(1, 2).contiguous())
    dx = I.conv_dgrad(dyd, wT, g, dims)
    assert I.tc_error() == 0
    B.check_dgrad(dx, dy, w.transpose(1, 2).contiguous(), g, acc[1])
    # wgrad (+dbias)
    dw, db = I.conv_wgrad(xd, dyd, g, want_bias=True)
    assert I.tc_error() == 0
    B.check_wgrad(dw, x, dy, g, acc[2], got_db=db)
    # MRA_CONV_ACCUMULATE: the kernels add into the caller's buffers (fused gradient accumulation)
    acc_w, acc_b = dw.clone(), db.clone()
    dw2, db2 = I.conv_wgrad(xd, dyd, g, want_bias=True, acc_dw=acc_w, acc_db=acc_b)
    assert dw2.data_ptr() == acc_w.data_ptr() and db2.data_ptr() == acc_b.data_ptr()
    B.check_wgrad(acc_w, x, dy, g, acc[2], got_db=acc_b, base_dw=dw, base_db=db, what="wgrad accumulate")


@pytest.mark.parametrize("case", CONVS, ids=gid)
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_conv_cuda_core_path(case, dtype):
    _check_conv(*case, dtype, expect_tc=False)


@pytest.mark.parametrize("case", TC_CONVS, ids=gid)
def test_conv_tcgen05_path(case):
    _check_conv(*case, torch.bfloat16, expect_tc=True)


def test_wgrad_cta_pair_path(monkeypatch):
    """wgrad_tc_kernel<true> (cta_group::2 pairs, used on G.rb at full size): force it on a shape the CPU reference can
    check, with enough K-blocks that stream-K ranges cross work-item boundaries; then the single-CTA kernel again."""
    case = (ConvGeom(256, 256, 3, 1, 0), (14, 12, 10), 2)
    monkeypatch.setenv("MRA_WGRAD_PAIR_MIN", "0")
    _check_conv(*case, torch.bfloat16, expect_tc=True)
    monkeypatch.setenv("MRA_WGRAD_NOPAIR", "1")
    _check_conv(*case, torch.bfloat16, expect_tc=True)


REPRO = [
    (ConvGeom(256, 256, 3, 1, 0), (34, 34, 34), 2),        # G.rb at full size: CTA pairs, every item over several units
    (ConvGeom(64, 128, 3, 2, 1), (64, 64, 64), 2),         # G.d1 at full size: four items, each over dozens of CTAs
]


@pytest.mark.parametrize("case", REPRO, ids=gid)
def test_wgrad_and_dbias_are_bit_reproducible(case):
    """A work item shared by several CTAs is added to dw in K order (wgrad_fixup_kernel) and the bias column sums in
    block order: the same inputs give the same dw and db bit for bit, also when they are added into a gradient."""
    I = ops.impl()
    g, dims, n = case
    x, _, _, dy = _conv_case(g, dims, n, torch.bfloat16)
    xd, dyd = x.cuda(), dy.cuda()
    dw, db = I.conv_wgrad(xd, dyd, g, want_bias=True)
    base_w, base_b = torch.randn_like(dw), torch.randn_like(db)
    acc = None
    for _ in range(3):
        w2, b2 = I.conv_wgrad(xd, dyd, g, want_bias=True)
        assert torch.equal(w2, dw) and torch.equal(b2, db)
        aw, ab = base_w.clone(), base_b.clone()
        I.conv_wgrad(xd, dyd, g, want_bias=True, acc_dw=aw, acc_db=ab)
        if acc is not None:
            assert torch.equal(aw, acc[0]) and torch.equal(ab, acc[1])
        acc = (aw, ab)
    assert I.tc_error() == 0
    if g.cin == 64:                                        # the fp64 reference of G.rb at 34^3 takes minutes on the host
        B.check_wgrad(dw, x, dy, g, "tc", got_db=db)
        B.check_wgrad(acc[0], x, dy, g, "tc", got_db=acc[1], base_dw=base_w, base_db=base_b, what="wgrad accumulate")


@pytest.mark.parametrize("case", TC_CONVS[:3], ids=gid)
def test_conv_same_shape_fp32_path(case):
    _check_conv(*case, torch.float32, expect_tc=False)


NORMS = [
    # (N, D, H, W, C, pad, act, residual_pad)
    (2, 6, 5, 7, 16, 1, R.ACT_RELU, -1),
    (1, 8, 8, 8, 64, 3, R.ACT_RELU, -1),
    (2, 4, 6, 5, 32, 1, R.ACT_NONE, 1),
    (2, 5, 5, 5, 24, 0, R.ACT_LRELU, -1),
    (1, 3, 4, 5, 4, 1, R.ACT_RELU, -1),        # scalar (C % 8 != 0) path
    (1, 2, 2, 2, 512, 0, R.ACT_LRELU, -1),     # tiny reduction, many channels
    (2, 4, 4, 4, 8, 0, R.ACT_NONE, 0),
    # row-streaming kernels (norm_stream.cuh): wide rows, deep pad folds, residual halo, re-cut rows, degenerate dims
    (1, 9, 7, 40, 64, 3, R.ACT_RELU, -1),
    (2, 10, 12, 33, 256, 1, R.ACT_NONE, 1),
    (1, 15, 15, 15, 512, 0, R.ACT_LRELU, -1),
    (2, 1, 1, 8, 16, 2, R.ACT_RELU, -1),
    (1, 3, 3, 1, 8, 1, R.ACT_RELU, -1),
    (3, 16, 16, 16, 128, 0, R.ACT_LRELU, -1),
    (1, 12, 12, 12, 256, 1, R.ACT_RELU, -1),
]


@pytest.mark.parametrize("case", NORMS, ids=lambda c: "x".join(map(str, c)))
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_inorm_act_pad(case, dtype):
    n, d, h, w, c, pad, act, rp = case
    I, ref = ops.impl(), R.RefImpl(torch.float64)
    gen = torch.Generator().manual_seed(1)
    x = (torch.randn((n, d, h, w, c), generator=gen) * 1.5 + 0.3).to(dtype)
    res = torch.randn((n, d + 2 * rp, h + 2 * rp, w + 2 * rp, c), generator=gen).to(dtype) if rp >= 0 else None
    gy = torch.randn((n, d + 2 * pad, h + 2 * pad, w + 2 * pad, c), generator=gen).to(dtype)
    rm, rv = torch.randn(c, generator=gen) * 0.1, 1 + 0.1 * torch.rand(c, generator=gen)
    tol = TOL[dtype]
    xd = x.cuda()
    st = I.inorm_stats(xd)
    st_ref = ref.inorm_stats(x)
    assert rel_l2(st.cpu(), st_ref) < 1e-5
    rmd, rvd = rm.cuda(), rv.cuda()
    y, mean, rstd = I.inorm_fwd(xd, st, res.cuda() if res is not None else None, pad, act, 0.2, rp,
                                running_mean=rmd, running_var=rvd)
    rm_r, rv_r = rm.clone().double(), rv.clone().double()
    y_ref, mean_ref, rstd_ref = ref.inorm_fwd(x.double(), st_ref, res.double() if res is not None else None, pad, act,
                                              0.2, rp, running_mean=rm_r, running_var=rv_r)
    assert rel_l2(y.cpu(), y_ref) < tol
    assert rel_l2(mean.cpu(), mean_ref) < 1e-5 and rel_l2(rstd.cpu(), rstd_ref) < 1e-5
    assert rel_l2(rmd.cpu(), rm_r) < 1e-5 and rel_l2(rvd.cpu(), rv_r) < 1e-5
    dx, dres = I.inorm_bwd(gy.cuda(), xd, mean, rstd, pad, act, 0.2, rp)
    dx_ref, dres_ref = ref.inorm_bwd(gy.double(), x.double(), mean_ref, rstd_ref, pad, act, 0.2, rp)
    assert rel_l2(dx.cpu(), dx_ref) < tol
    if rp >= 0:
        assert rel_l2(dres.cpu(), dres_ref) < tol
    # eval mode (running statistics)
    y2, m2, r2 = I.inorm_fwd(xd, st, None, pad, act, 0.2, -1, running_mean=rmd, running_var=rvd, use_running=True)
    y2_ref, _, _ = ref.inorm_fwd(x.double(), st_ref, None, pad, act, 0.2, -1, running_mean=rm_r, running_var=rv_r,
                                 use_running=True)
    assert rel_l2(y2.cpu(), y2_ref) < tol


def test_norm_matches_torch_instance_norm_module():
    """End-to-end against the reference's own layer composition (networks3D.py:232-243):
    ReplicationPad3d(1) o ReLU o InstanceNorm3d, forward and backward through autograd."""
    import torch.nn.functional as F
    I = ops.impl()
    gen = torch.Generator().manual_seed(3)
    x = torch.randn((2, 16, 6, 6, 6), generator=gen, dtype=torch.float64, requires_grad=True)
    rm, rv = torch.zeros(16, dtype=torch.float64), torch.ones(16, dtype=torch.float64)
    y = F.pad(F.relu(F.instance_norm(x, rm, rv, use_input_stats=True, momentum=0.1, eps=1e-5)), (1,) * 6, mode="replicate")
    gy = torch.randn(y.shape, generator=gen, dtype=torch.float64)
    y.backward(gy)
    xl = x.detach().permute(0, 2, 3, 4, 1).contiguous().float().cuda()
    rmd, rvd = torch.zeros(16).cuda(), torch.ones(16).cuda()
    st = I.inorm_stats(xl)
    yl, mean, rstd = I.inorm_fwd(xl, st, None, 1, ops.ACT_RELU, running_mean=rmd, running_var=rvd)
    assert rel_l2(yl.cpu().permute(0, 4, 1, 2, 3), y.detach()) < 1e-5
    assert rel_l2(rmd.cpu(), rm) < 1e-5 and rel_l2(rvd.cpu(), rv) < 1e-5
    dx, _ = I.inorm_bwd(gy.permute(0, 2, 3, 4, 1).contiguous().float().cuda(), xl, mean, rstd, 1, ops.ACT_RELU)
    assert rel_l2(dx.cpu().permute(0, 4, 1, 2, 3), x.grad) < 1e-4


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_pad_act_standalone(dtype):
    I, ref = ops.impl(), R.RefImpl(torch.float64)
    gen = torch.Generator().manual_seed(2)
    for c in (1, 8):
        x = torch.randn((2, 5, 4, 6, c), generator=gen).to(dtype)
        y = I.reppad_fwd(x.cuda(), 3)
        assert torch.equal(y.cpu(), ref.reppad_fwd(x, 3))
        gy = torch.randn(y.shape, generator=gen).to(dtype)
        assert rel_l2(I.reppad_bwd(gy.cuda(), 3).cpu(), ref.reppad_bwd(gy.double(), 3)) < TOL[dtype]
    x = torch.randn((3, 4, 5, 6, 7), generator=gen).to(dtype)
    for act in (R.ACT_RELU, R.ACT_LRELU, R.ACT_TANH, R.ACT_SIGMOID):
        y = I.act_fwd(x.cuda(), act, 0.2)
        assert rel_l2(y.cpu(), ref.act_fwd(x.double(), act, 0.2)) < TOL[dtype]
        dx = I.act_bwd(x.cuda(), y, act, 0.2)
        assert rel_l2(dx.cpu(), ref.act_bwd(x.double(), y.cpu().double(), act, 0.2)) < TOL[dtype]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_dropout_mask_scale(dtype):
    """mra_mask_scale (nn.Dropout in training mode): exact against the oracle for a given keep mask, and through
    functional.DropoutFn: 1/(1-p) scaling, the backward reuses the forward's mask."""
    from mra_gan_b200 import functional as MF
    I, ref = ops.impl(), R.RefImpl(torch.float64)
    gen = torch.Generator().manual_seed(4)
    x = torch.randn((2, 5, 6, 7, 24), generator=gen).to(dtype)
    keep = (torch.rand(x.shape, generator=gen) > 0.5).to(torch.uint8)
    y = I.mask_scale(x.cuda(), keep.cuda(), 2.0)
    assert torch.equal(y.cpu(), ref.mask_scale(x, keep, 2.0))
    xd = x.cuda().requires_grad_(True)
    z = MF.DropoutFn.apply(xd, 0.5)
    kept = z != 0
    assert 0.4 < float(kept.float().mean()) < 0.6
    assert torch.equal(z[kept], (2.0 * xd.detach().float()[kept]).to(dtype))
    z.float().sum().backward()
    assert torch.equal(xd.grad != 0, kept)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_losses(dtype):
    I, ref = ops.impl(), R.RefImpl(torch.float64)
    gen = torch.Generator().manual_seed(4)
    a = torch.randn((2, 14, 14, 14, 1), generator=gen).to(dtype)
    b = torch.randn((2, 14, 14, 14, 1), generator=gen).to(dtype)
    p = torch.rand((2, 6, 6, 6, 1), generator=gen).clamp(1e-3, 1 - 1e-3).to(dtype)
    gout = torch.tensor(0.7)
    for kind, aa, bb, tgt in ((R.LOSS_L1, a, b, 0.0), (R.LOSS_MSE_CONST, a, None, 1.0), (R.LOSS_MSE_CONST, a, None, 0.0),
                              (R.LOSS_BCE_CONST, p, None, 1.0), (R.LOSS_BCE_CONST, p, None, 0.0)):
        got = I.loss_fwd(kind, aa.cuda(), bb.cuda() if bb is not None else None, tgt)
        want = ref.loss_fwd(kind, aa.double(), bb.double() if bb is not None else None, tgt)
        assert float(got) == pytest.approx(float(want), rel=1e-5)
        da = I.loss_bwd(kind, aa.cuda(), bb.cuda() if bb is not None else None, tgt, gout.cuda(), 3.0 / aa.numel())
        da_ref = ref.loss_bwd(kind, aa.double(), bb.double() if bb is not None else None, tgt, gout.double(), 3.0 / aa.numel())
        assert rel_l2(da.cpu(), da_ref) < TOL[dtype]
    s = I.corr_sums(a.cuda(), b.cuda())
    assert rel_l2(s.cpu(), ref.corr_sums(a, b)) < 1e-6


def test_adam_matches_torch_optim():
    I = ops.impl()
    gen = torch.Generator().manual_seed(5)
    # > 48 tensors: several launches; sizes that are not multiples of 4 exercise the tail of the 16-byte path
    shapes = [(27, 16, 16), (16,), (343, 8, 1), (5000,), (1,), (1023,), (7,)] * 9
    ps = [torch.randn(s, generator=gen) for s in shapes]
    ref_p = [p.clone().requires_grad_(True) for p in ps]
    opt = torch.optim.Adam(ref_p, lr=2e-4, betas=(0.5, 0.999))
    dp = [p.cuda() for p in ps]
    # a parameter that is only 4-byte aligned (a view one element into its buffer): the scalar path
    mis = torch.zeros(ps[3].numel() + 1, device="cuda")
    mis[1:].copy_(ps[3].cuda())
    dp[3] = mis[1:]
    assert dp[3].data_ptr() % 16 == 4
    m = [torch.zeros_like(p) for p in dp]
    v = [torch.zeros_like(p) for p in dp]
    sh = [torch.empty_like(p, dtype=torch.bfloat16) if i % 2 == 0 else None for i, p in enumerate(dp)]
    for step in range(1, 4):
        gs = [torch.randn(s, generator=gen) * (0.1 if step < 3 else 1e-6) for s in shapes]
        for p, g in zip(ref_p, gs):
            p.grad = g.clone()
        opt.step()
        I.adam_step(dp, [g.cuda() for g in gs], m, v, sh, 2e-4, 0.5, 0.999, 1e-8, step)
        for a, b in zip(dp, ref_p):
            assert float((a.cpu() - b.detach()).abs().max()) < 5e-7          # 1 fp32 ulp at |p| in [2, 4) is 2.4e-7
    for a, s in zip(dp, sh):
        if s is not None:
            assert torch.equal(s.cpu(), a.cpu().to(torch.bfloat16))


@pytest.mark.parametrize("dtype,ca,cb", [(torch.bfloat16, 64, 128), (torch.bfloat16, 8, 8), (torch.bfloat16, 4, 12),
                                         (torch.float32, 16, 8), (torch.float32, 3, 5)])
def test_cat2_act(dtype, ca, cb):
    """UNet skip: act(cat([a, b], C)) written in one pass and its backward (networks3D.py:339-343 + the parent's ReLU)."""
    I, ref = ops.impl(), R.RefImpl(torch.float32)
    gen = torch.Generator().manual_seed(9)
    a = torch.randn((2, 5, 6, 7, ca), generator=gen).to(dtype)
    b = torch.randn((2, 5, 6, 7, cb), generator=gen).to(dtype)
    go = torch.randn((2, 5, 6, 7, ca + cb), generator=gen).to(dtype)
    for act, slope in ((1, 0.0), (2, 0.2), (0, 0.0)):
        out = I.cat2_act_fwd(a.cuda(), b.cuda(), act, slope)
        want = ref.cat2_act_fwd(a, b, act, slope)
        assert torch.equal(out.cpu(), want)
        da, db = I.cat2_act_bwd(go.cuda(), out, ca, act, slope)
        wa, wb = ref.cat2_act_bwd(go, want, ca, act, slope)
        assert torch.equal(da.cpu(), wa) and torch.equal(db.cpu(), wb)
        da, db = I.cat2_act_bwd(go.cuda(), out, ca, act, slope, (False, True))
        assert da is None and torch.equal(db.cpu(), wb)


NSTATS = [
    # geom, in_dims (= shape of the norm's stored output), N, norm act, slope      -> kernel
    (ConvGeom(256, 256, 3, 1, 0), (10, 10, 10), 2, 1, 0.0),             # res-block conv2 dgrad: gather_halo (2D / flat tiles)
    (ConvGeom(256, 256, 3, 1, 0), (34, 34, 34), 2, 1, 0.0),             # the same at config-2 size (split tail items)
    (ConvGeom(64, 128, 3, 2, 1), (16, 16, 16), 2, 1, 0.0),              # G.d1 dgrad: merged phases, paired (n_tile 64)
    (ConvGeom(64, 128, 3, 2, 1), (128, 128, 128), 1, 1, 0.0),           # ... at full size (64 ch x 128^3)
    (ConvGeom(128, 256, 3, 2, 1), (16, 16, 16), 2, 1, 0.0),             # G.d2 dgrad: merged 8 phases
    (ConvGeom(128, 64, 3, 2, 1, True, 1), (8, 8, 8), 2, 1, 0.0),        # G.u2 dgrad (ConvTranspose3d): strided gather
    (ConvGeom(64, 1, 7, 1, 0), (22, 22, 22), 2, 1, 0.0),                # head dgrad: column kernel, dual planes
    (ConvGeom(128, 256, 4, 2, 1), (16, 16, 16), 2, 2, 0.2),             # D.3 dgrad, LeakyReLU(0.2)
    (ConvGeom(256, 512, 4, 1, 1), (9, 9, 9), 2, 2, 0.2),                # D.4 dgrad (zero-padded stride 1)
    (ConvGeom(256, 256, 3, 1, 0), (10, 10, 10), 1, 0, 0.0),             # no activation between norm and conv
]


@pytest.mark.parametrize("case", NSTATS, ids=lambda c: "%d-%d_k%ds%d%s_%s_n%d_act%d" % (
    c[0].cin, c[0].cout, c[0].k, c[0].stride, "T" if c[0].transposed else "", "x".join(map(str, c[1])), c[2], c[3]))
def test_conv_dgrad_norm_backward_statistics(case):
    """mra_conv3d_dgrad_nstats: dx is bit-identical to the plain dgrad, and sums[n][c] = {sum dx act'(y), sum dx y}
    over every (padded) position -- what the statistics pass of the norm backward computes from (dx, x) -- here checked
    in fp64 from the stored dx (bf16) and y."""
    g, dims, n, act, slope = case
    I = ops.impl()
    gen = torch.Generator(device="cuda").manual_seed(3)
    out_dims = g.out_dims(dims)
    dy = torch.randn((n,) + out_dims + (g.cout,), generator=gen, device="cuda").to(torch.bfloat16)
    w = (torch.randn((g.taps, g.cout, g.cin), generator=gen, device="cuda") / (g.taps * g.cout) ** 0.5).to(torch.bfloat16)
    wT = I.pack_weight_t(w, torch.bfloat16)
    xh = torch.randn((n,) + dims + (g.cin,), generator=gen, device="cuda")
    ns = {0: 1.0, 1: 0.0}.get(act, slope)
    y = torch.where(xh > 0, xh, xh * ns).to(torch.bfloat16)
    assert I.conv_dgrad_nstats_supported(g, n, dims, torch.bfloat16)
    low, ws = I.conv_shared_workspace(g, n, dims, torch.bfloat16, "cuda")
    kw = dict(ws=ws) if low else {}
    dx_ref = I.conv_dgrad(dy, wT, g, dims, **kw)
    dx, sums = I.conv_dgrad_nstats(dy, wT, g, dims, y, act, slope, **kw)
    assert I.tc_error() == 0
    assert torch.equal(dx, dx_ref)
    y64 = y.double()
    wgt = torch.where(y64 > 0, torch.ones_like(y64), torch.full_like(y64, ns))
    cnt = dx[0, ..., 0].numel()
    if dx.numel() <= 4_000_000:
        # small case: the oracle's UNROUNDED fp32 dgrad of the same bf16 operands -- only the summation order differs
        d64 = R.RefImpl(torch.float32).conv_dgrad(dy.float().cpu(), wT.float().cpu(), g, dims).double().cuda()
        tol = lambda a: 3e-5 * a + 1e-9
    else:
        # full size: the stored bf16 dx; the epilogue sums the fp32 accumulators, so the two differ by the rounding of
        # dx (relative 2^-8 at most, random sign): |diff| ~ 2^-8 sum|term| / sqrt(count); a lost or doubled tile would
        # be >= sum|term| / tiles
        d64 = dx.double()
        tol = lambda a: 10 * 2.0 ** -8 * a / cnt ** 0.5 + 1e-6 * a + 1e-9
    s0, s1 = (d64 * wgt).sum((1, 2, 3)), (d64 * y64).sum((1, 2, 3))
    a0, a1 = (d64 * wgt).abs().sum((1, 2, 3)), (d64 * y64).abs().sum((1, 2, 3))
    assert bool(((sums[..., 0] - s0).abs() <= tol(a0)).all()), float(((sums[..., 0] - s0).abs() / a0).max())
    assert bool(((sums[..., 1] - s1).abs() <= tol(a1)).all()), float(((sums[..., 1] - s1).abs() / a1).max())


def test_norm_backward_with_statistics_from_the_dgrad_epilogue_matches_two_pass():
    """End to end through autograd: (InstanceNorm -> ReLU -> pad) -> conv with the NormBwdLink (statistics from the conv's
    dgrad epilogue, apply pass only) against the same program with MRA_NORM_BWD_FUSED off (two-pass norm backward)."""
    from mra_gan_b200 import networks3D as N3
    N3.set_default_compute_dtype(torch.bfloat16)
    torch.manual_seed(0)
    seq = torch.nn.Sequential(N3.Conv3d(64, 256, 3, 1, 1), N3.InstanceNorm3d(256), N3.ReLU(True), N3.ReplicationPad3d(1),
                              N3.Conv3d(256, 256, 3, 1, 0), N3.InstanceNorm3d(256), N3.ReLU(True),
                              N3.Conv3d(256, 128, 3, 2, 1)).cuda()
    prog = N3.compile_program(seq)
    x = torch.randn(2, 12, 12, 12, 64, device="cuda").to(torch.bfloat16)
    outs = []
    for fused in (True, True, False):               # the first pass warms the weight caches (pack / convert launches)
        N3._FUSE_NORM_BWD = fused
        try:
            for p in seq.parameters():
                p.grad = None
            xi = x.clone().requires_grad_(True)
            n0 = ops.impl().launch_count()
            y = N3.run_program(prog, xi)
            y.float().square().mean().backward()
            outs.append((xi.grad.float(), [p.grad.float().clone() for p in seq.parameters() if p.grad is not None],
                         ops.impl().launch_count() - n0))
        finally:
            N3._FUSE_NORM_BWD = True
    outs = outs[1:]
    assert outs[0][2] < outs[1][2]                          # the linked norms skip their statistics launch
    assert rel_l2(outs[0][0], outs[1][0]) < 5e-3
    for a, b in zip(outs[0][1], outs[1][1]):
        if float(b.abs().max()) > 0:
            assert rel_l2(a, b) < 5e-3


def test_fused_adam_graph_replay_runs_ahead_of_the_device():
    """VERDICT r1 weak #3 / ADVICE (medium): the captured optimiser step must advance by exactly ONE Adam step per
    replay even when the host runs many replays ahead of the device (no sync in between; a busy-wait kernel in front
    of every replay makes sure it does).  The step counter and both bias corrections live on the device
    (mra_adam_advance), so 8 un-synchronised replays == 8 eager, synchronised steps bit for bit, and both sit on
    torch.optim.Adam (fp32) to 1e-6 -- sqrt(1 - 0.999^t) changes by 41 % between t = 1 and t = 2, so a step that read a
    later step's corrections would be off by far more."""
    from mra_gan_b200.optim import FusedAdam
    gen = torch.Generator().manual_seed(11)
    shapes = [(27, 16, 16), (16,), (343, 8, 1), (5000,)]
    init = [torch.randn(s, generator=gen) * 0.02 for s in shapes]
    grads = [[torch.randn(s, generator=gen) * 0.1 for s in shapes] for _ in range(9)]

    def make():
        ps = [torch.nn.Parameter(p.clone().cuda()) for p in init]
        for p in ps:
            p.grad = torch.zeros_like(p)
        return ps, FusedAdam(ps, lr=2e-4, betas=(0.5, 0.999))

    # eager, synchronised after every step
    pe, oe = make()
    for gs in grads:
        for p, g in zip(pe, gs):
            p.grad.copy_(g.cuda())
        oe.step()
        torch.cuda.synchronize()
    # graph: one eager step, then capture, then replays fed from a device-side queue of gradients with NO host sync
    pg, og = make()
    gq = [torch.stack([gs[i] for gs in grads]).cuda() for i in range(len(shapes))]     # [step][...] per tensor
    idx = torch.zeros((), dtype=torch.long, device="cuda")

    def load_grads():
        for p, q in zip(pg, gq):
            p.grad.copy_(q.index_select(0, idx.reshape(1))[0])
        idx.add_(1)

    load_grads(); og.step()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        load_grads(); og.step()
    graph.replay()                                   # executes step 2 (capture only records)
    for _ in range(len(grads) - 2):
        torch.cuda._sleep(20_000_000)                # ~10 ms of device work queued in front: the host runs ahead
        og.advance_host_state()
        graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(pg, pe):
        assert torch.equal(a.detach(), b.detach())
    assert og.state[pg[0]]["step"] == len(grads)
    # torch.optim.Adam on the CPU, fp32
    pr = [p.clone().requires_grad_(True) for p in init]
    ot = torch.optim.Adam(pr, lr=2e-4, betas=(0.5, 0.999))
    for gs in grads:
        for p, g in zip(pr, gs):
            p.grad = g.clone()
        ot.step()
    for a, b in zip(pg, pr):
        assert float((a.detach().cpu() - b.detach()).abs().max()) < 1e-6
    # a learning-rate change between replays reaches the device before the next replay
    for group in og.param_groups + ot.param_groups + oe.param_groups:
        group["lr"] = 5e-5
    for p, g in zip(pr, grads[0]):
        p.grad = g.clone()
    ot.step()
    idx.zero_()
    og.advance_host_state()
    graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(pg, pr):
        assert float((a.detach().cpu() - b.detach()).abs().max()) < 1e-6


def test_sliding_window_helpers():
    I, ref = ops.impl(), R.RefImpl()
    gen = torch.Generator().manual_seed(6)
    vol = torch.rand((20, 18, 11), generator=gen) * 255
    lab, wt = torch.zeros_like(vol), torch.zeros_like(vol)
    labd, wtd, vold = lab.cuda(), wt.cuda(), vol.cuda()
    for (i0, j0, k0) in ((0, 0, 0), (12, 10, 3), (4, 2, 1)):
        pr = ref.window_extract(vol, i0, j0, k0, (8, 8, 8), torch.float32)
        pd = I.window_extract(vold, i0, j0, k0, (8, 8, 8), torch.float32)
        assert torch.equal(pd.cpu(), pr)
        ref.window_accumulate(pr * 0.5, lab, wt, i0, j0, k0)
        I.window_accumulate(pd * 0.5, labd, wtd, i0, j0, k0)
    assert torch.allclose(labd.cpu(), lab, atol=1e-4) and torch.equal(wtd.cpu(), wt)
    lab += 1; wt += 1; labd += 1; wtd += 1
    ref.window_finalize(lab, wt)
    I.window_finalize(labd, wtd)
    assert torch.allclose(labd.cpu(), lab, atol=1e-4)


KSPLIT = [
    (ConvGeom(512, 512, 4, 2, 1), (8, 8, 8), 4),               # UNet-7 d5 at config 4's per-GPU batch
    (ConvGeom(512, 512, 4, 2, 1), (2, 2, 2), 4),               # d7: 2^3 -> 1^3, four output positions
    (ConvGeom(1024, 512, 4, 2, 1, True, 0), (2, 2, 2), 2),     # u6 (its dgrad is the direct stride-2 form)
    (ConvGeom(256, 512, 4, 2, 1), (16, 16, 16), 2),            # d4
    (ConvGeom(256, 128, 3, 2, 1), (8, 8, 8), 1),               # 27 taps: uneven tap ranges (3,3,4,3,3,4,3,4)
]


@pytest.mark.parametrize("case", KSPLIT, ids=gid)
def test_split_k_gather_matches_unsplit_and_oracle(case, monkeypatch):
    """Launches with a handful of output tiles and a long reduction run as 8 tap ranges with fp32 partial sums in the
    caller's workspace (conv_tc_halo.cuh: run_gather_ksplit).  Against the unsplit kernel (MRA_GATHER_NOKSPLIT) and the fp64
    oracle, for the op whose plan is the direct stride-2 form: fprop of a Conv3d, dgrad of a ConvTranspose3d."""
    import ctypes as C
    g, dims, n = case
    I = ops.impl()
    x, w, b, dy = _conv_case(g, dims, n, torch.bfloat16, seed=5)
    xd, wd, bd, dyd = x.cuda(), w.cuda(), b.cuda(), dy.cuda()
    which = 1 if g.transposed else 0
    d = I._conv_desc(g, n, dims, g.out_dims(dims), ops.MRA_BF16)
    assert int(I.L.mra_conv3d_workspace_size(C.byref(d), which)) > 0, "case is expected to take the split-K path"
    if not g.transposed:
        y, st = I.conv_fprop(xd, wd, bd, g, want_stats=True)
        y3, _ = I.conv_fprop(xd, wd, None, g, act=ops.ACT_LRELU, slope=0.2)
        monkeypatch.setenv("MRA_GATHER_NOKSPLIT", "1")
        assert int(I.L.mra_conv3d_workspace_size(C.byref(d), which)) == 0
        y2, st2 = I.conv_fprop(xd, wd, bd, g, want_stats=True)
        pre, mag = B.fprop_ref(x, w, b, g)
        B.check_output(y, pre, mag, "tc", what="split fprop")
        B.check_output(y2, pre, mag, "tc", what="unsplit fprop")
        B.check_stats(st, pre, mag, torch.bfloat16, "tc", "split statistics")
        B.check_stats(st2, pre, mag, torch.bfloat16, "tc", "unsplit statistics")
        B.check_fprop(y3, x, w, None, g, "tc", R.ACT_LRELU, 0.2, what="split fprop+lrelu")
    else:
        wT = I.pack_weight_t(wd, torch.bfloat16)
        dx = I.conv_dgrad(dyd, wT, g, dims)
        monkeypatch.setenv("MRA_GATHER_NOKSPLIT", "1")
        dx2 = I.conv_dgrad(dyd, wT, g, dims)
        B.check_dgrad(dx, dy, w.transpose(1, 2).contiguous(), g, "tc", "split dgrad")
        B.check_dgrad(dx2, dy, w.transpose(1, 2).contiguous(), g, "tc", "unsplit dgrad")
    assert I.tc_error() == 0


DEAD_PLANES = [
    (ConvGeom(256, 256, 3, 1, 0), (14, 12, 10), 2),            # G.rb dgrad: 14^3-ish padded gradient, flat tiles, CTA pairs
    (ConvGeom(256, 256, 3, 1, 0), (9, 10, 10), 1),             # odd plane count: the last pair's partner plane does not exist
    (ConvGeom(256, 512, 4, 1, 1), (9, 9, 9), 2),               # D.4: zero padding, dead planes in fprop AND dgrad
    (ConvGeom(64, 64, 3, 1, 1), (9, 7, 5), 1),
]


@pytest.mark.parametrize("mode", ["pair", "single"])
@pytest.mark.parametrize("case", DEAD_PLANES, ids=gid)
def test_halo_dead_plane_skipping_is_bit_identical(case, mode, monkeypatch):
    """gather_halo_kernel skips input planes that lie outside the A tensor for every tile of a work item (conv_tc_halo.cuh:
    halo_plane_live): no plane load, no weight slabs, no MMAs.  The skipped MMAs multiply TMA zero fill, so the result
    must be the same bits as with MRA_HALO_NOSKIP=1 (epilogue statistics: up to the order of fp64 atomics) and match the
    fp64 oracle."""
    g, dims, n = case
    I = ops.impl()
    if mode == "single":
        monkeypatch.setenv("MRA_GATHER_MODE", "single")
    x, w, b, dy = _conv_case(g, dims, n, torch.bfloat16, seed=11)
    xd, wd, bd, dyd = x.cuda(), w.cuda(), b.cuda(), dy.cuda()
    wT = I.pack_weight_t(wd, torch.bfloat16)
    y, st = I.conv_fprop(xd, wd, bd, g, want_stats=True)
    dx = I.conv_dgrad(dyd, wT, g, dims)
    monkeypatch.setenv("MRA_HALO_NOSKIP", "1")
    y0, st0 = I.conv_fprop(xd, wd, bd, g, want_stats=True)
    dx0 = I.conv_dgrad(dyd, wT, g, dims)
    assert I.tc_error() == 0
    assert bool((y.float() == y0.float()).all()) and bool((dx.float() == dx0.float()).all())
    assert torch.allclose(st, st0, rtol=1e-9, atol=1e-9)        # fp64 atomics: the order of the CTAs' adds is free
    B.check_fprop(y, x, w, b, g, "tc", got_stats=st)
    B.check_dgrad(dx, dy, w.transpose(1, 2).contiguous(), g, "tc")


DUAL_CASES = [
    # (geom, in_dims, n, which)        launches whose tile count per plane is even: eligible for dual items
    (ConvGeom(256, 256, 3, 1, 0), (18, 18, 18), 1, 0),         # fprop, 2D tiles (2 per plane)
    (ConvGeom(256, 256, 3, 1, 0), (18, 18, 18), 3, 0),
    (ConvGeom(256, 256, 3, 1, 0), (12, 12, 12), 2, 1),         # dgrad
    (ConvGeom(256, 256, 3, 1, 0), (34, 34, 34), 2, 0),         # the bench's G.rb fprop (split tail items) ...
    (ConvGeom(256, 256, 3, 1, 0), (34, 34, 34), 2, 1),         # ... and dgrad (flat tiles, dead planes)
    (ConvGeom(256, 256, 3, 1, 0), (34, 34, 34), 3, 1),
]


@pytest.mark.parametrize("case", DUAL_CASES, ids=lambda c: gid(c[:3]) + "_" + "fd"[c[3]])
def test_halo_dual_items_match_single_items_and_oracle(case, monkeypatch):
    """MRA_HALO_DUAL=1: a work item of gather_halo_kernel is two position tiles x 128 channels (every weight slab feeds two
    tiles) instead of one tile x 256.  Same sums in another order: against the default kernel to bf16 rounding, against the
    fp64 oracle where it finishes in seconds; epilogue statistics (fprop) and norm-backward statistics (dgrad) included."""
    g, dims, n, which = case
    I = ops.impl()
    small = dims[0] <= 18
    x, w, b, dy = _conv_case(g, dims, n, torch.bfloat16, seed=3)
    xd, wd, bd, dyd = x.cuda(), w.cuda(), b.cuda(), dy.cuda()
    wT = I.pack_weight_t(wd, torch.bfloat16)

    def run():
        if which == 0:
            y, st = I.conv_fprop(xd, wd, bd, g, want_stats=True)
            return y, st
        dx = I.conv_dgrad(dyd, wT, g, dims)
        dx2, sums = I.conv_dgrad_nstats(dyd, wT, g, dims, xd, ops.ACT_RELU, 0.0)
        assert bool((dx.float() == dx2.float()).all())
        return dx, sums

    monkeypatch.delenv("MRA_HALO_DUAL", raising=False)
    a0, s0 = run()
    monkeypatch.setenv("MRA_HALO_DUAL", "1")
    words = ops.schedule_describe(g, n, dims, which)
    assert words[0] == 1 and words[1] == 1 and words[2 + 17] == 2, "case is expected to run as dual items"
    a1, s1 = run()
    assert I.tc_error() == 0
    assert rel_l2(a1.float().cpu(), a0.float().cpu()) < 4e-3
    assert rel_l2(s1.cpu(), s0.cpu()) < 1e-3
    if small:
        if which == 0:
            B.check_fprop(a1, x, w, b, g, "tc", got_stats=s1, what="dual-item fprop")
        else:
            B.check_dgrad(a1, dy, w.transpose(1, 2).contiguous(), g, "tc", "dual-item dgrad")
