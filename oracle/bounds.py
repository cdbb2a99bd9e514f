"""Per-element error bounds for the convolution family (TEST INFRASTRUCTURE, next to ops_ref.py).

A global rel-L2 over a whole tensor lets a bug that touches a small part of it pass: a tap dropped on the last w
column, one 64-channel K chunk lost on one tile, a tile's statistics counted twice.  The checks here bound EVERY
element by what the arithmetic of the kernels allows.  For an op with fp64 reference ``ref`` (``RefImpl(float64)`` on
the operands as stored) and magnitude ``mag`` (the same op on the absolute values of the operands):

    |got - act(ref + b)| <= r_out * |act(ref + b)| + L_act * CU[acc] * mag

* ``r_out``: the rounding of the stored output, 2^-8 for bf16 (round to nearest, 8 significant bits: 2^-9 for the
  rounding, the other 2^-9 absorbs the rounding of fp32 activations near a bf16 tie), 0 for fp32 outputs.
* ``L_act``: the Lipschitz constant of the fused activation (1; 1/4 for the sigmoid): an accumulator error e moves the
  activated output by at most L_act * e.
* ``CU[acc]``: the relative accumulation error, one constant per accumulation type (see CU below).

Epilogue statistics are checked per (n, c), the sum and the sum of squares separately, against fp64 sums of the
unrounded ``ref + b``: the bound of a sum is the sum of the element bounds, that of a sum of squares
sum_i (2 |y_i| + bound_i) bound_i.  Bias gradients are checked per channel against the fp64 column sum with the fp32
summation constant.  Every check raises ``BoundError`` naming the worst element and returns the largest error / bound
ratio it saw (< 1 on success) so that tests can print it.
"""
import torch

from . import ops_ref as R

# Relative accumulation error, times mag, one constant per accumulation type.
#
# "tc" (tcgen05.mma, bf16 operands, fp32 accumulator in tensor memory).  Products of two bf16 values are exact in fp32.
#   The MMA adds each K=16 block of them to the accumulator after aligning the addends to the largest exponent, and
#   may drop the bits shifted out (truncation, not rounding): a step loses less than 2^-22 of the magnitude it adds,
#   which is at most the partial magnitude of the reduction so far, hence less than 2^-22 mag.  Linear growth over
#   K/16 <= 2^10 steps bounds the total by 2^-12 mag.  Longer reductions (wgrad over many positions, split-K and
#   stream-K pieces added in fp32) have zero-mean operands here, whose step errors carry independent signs and grow
#   as the square root of the step count: 2^-12 still holds with a wide margin.
# "tc_bf16" (the channel-expanded lowerings of conv_special.cuh whose tensor-core result is a bf16 PARTIAL sum, summed
#   again afterwards: head fprop and stem dgrad store Z, one partial per folded (kh, kw); the im2col dgrad and the
#   ConvTranspose3d(C -> 1) fprop store dE, one partial per tap, before col2im).  Each partial is rounded to 2^-9 of
#   its own magnitude and the partials' magnitudes add up to at most mag: 2^-9 mag, on top of the "tc" term.
# "fma" (CUDA-core kernels: sequential fp32 fmaf chains; column sums in fp32 partials added in order).  Each step
#   rounds to 2^-24 of the partial sum, which is at most the magnitude so far: linear growth bounds it by K 2^-24 mag,
#   i.e. 2^-17 mag for K <= 2^7; for longer zero-mean reductions the partial sums are ~sqrt(K) smaller than mag and the
#   independently signed roundings add as a square root, which keeps the error near 2^-24 mag at any K.
# "fp64": the oracle checking itself (CPU self-tests of the full-size checker): fp64 sums, but the oracle returns dw
#   in fp32, rounded to 2^-24 of |dw| <= mag.
CU = {"tc": 2.0 ** -12, "tc_bf16": 2.0 ** -9 + 2.0 ** -12, "fma": 2.0 ** -17, "fp64": 2.0 ** -23}
R_OUT = {torch.bfloat16: 2.0 ** -8, torch.float32: 0.0, torch.float64: 0.0}
L_ACT = {R.ACT_NONE: 1.0, R.ACT_RELU: 1.0, R.ACT_LRELU: 1.0, R.ACT_TANH: 1.0, R.ACT_SIGMOID: 0.25}

_REF = R.RefImpl(torch.float64)


class BoundError(AssertionError):
    pass


def acc_type(dtype, tensor_cores, lowering=0, which=0):
    """The accumulation type of op ``which`` (0 fprop, 1 dgrad, 2 wgrad) of a layer: fmaf on the CUDA-core kernels,
    tcgen05 on the tensor cores, with a bf16 partial sum for the ops of a lowering that sum the tensor-core result
    again (``lowering`` = mra_conv3d_lowering: 1 stem, 2 head / ConvTranspose3d(C -> 1), 3 im2col)."""
    if dtype == torch.float64:
        return "fp64"
    if not tensor_cores:
        return "fma"
    partial = (lowering in (1, 3) and which == 1) or (lowering == 2 and which == 0)
    return "tc_bf16" if partial else "tc"


# ---------------------------------------------------------------------------------------------------------------
# fp64 references and magnitudes (channels-last, [taps][Cout][Cin] weights, as the library stores them)
# ---------------------------------------------------------------------------------------------------------------
def _d(t):
    return t.detach().cpu().double()


def fprop_ref(x, w, bias, g):
    """(ref + b, mag) of conv_fprop, both fp64 (N, D, H, W, Cout); pre-activation."""
    x, w = _d(x), _d(w)
    ref, _ = _REF.conv_fprop(x, w, None if bias is None else _d(bias), g)
    mag, _ = _REF.conv_fprop(x.abs(), w.abs(), None, g)
    return ref, mag


def dgrad_ref(dy, wT, g, in_dims):
    dy, wT = _d(dy), _d(wT)
    return _REF.conv_dgrad(dy, wT, g, in_dims), _REF.conv_dgrad(dy.abs(), wT.abs(), g, in_dims)


def wgrad_ref(x, dy, g):
    """(dw, mag) fp64 [taps][Cout][Cin]."""
    x, dy = _d(x), _d(dy)

    def wgrad(a, b):                       # RefImpl.conv_wgrad, without its fp32 result
        w0 = R.unpack_weight(torch.zeros((g.taps, g.cout, g.cin), dtype=torch.float64), g.k, g.transposed)
        gw = _REF._conv_backward(R.to_ncdhw(b), R.to_ncdhw(a).contiguous(), w0, g, [False, True, False])[1]
        return R.pack_weight(gw, g.transposed)
    return wgrad(x, dy), wgrad(x.abs(), dy.abs())


def _act64(v, act, slope):
    return R._act(v, act, slope)


# ---------------------------------------------------------------------------------------------------------------
# element checks
# ---------------------------------------------------------------------------------------------------------------
def _worst(ratio, names):
    i = int(torch.argmax(torch.nan_to_num(ratio, nan=float("inf"))))
    idx = []
    for s in reversed(ratio.shape):
        idx.append(i % s)
        i //= s
    idx = tuple(reversed(idx))
    return idx, "(" + ", ".join("%s=%d" % (n, v) for n, v in zip(names, idx)) + ")"


def _ratio(err, bound):
    return torch.where(bound > 0, err / torch.where(bound > 0, bound, torch.ones_like(bound)),
                       torch.where(err > 0, torch.full_like(err, float("inf")), torch.zeros_like(err)))


def check_elements(got, want, bound, what, names):
    """|got - want| <= bound element by element; returns the worst ratio."""
    got = _d(got)
    assert got.shape == want.shape == bound.shape, (what, tuple(got.shape), tuple(want.shape))
    err = (got - want).abs()
    ratio = _ratio(err, bound)
    if ratio.numel() == 0:
        return 0.0
    idx, where = _worst(ratio, names)
    worst = float(ratio[idx])
    if not worst <= 1.0:
        raise BoundError("%s: element %s got %.6g, want %.6g, |err| %.3g > bound %.3g (ratio %.3g)" % (
            what, where, float(got[idx]), float(want[idx]), float(err[idx]), float(bound[idx]), worst))
    return worst


def output_bound(pre, mag, out_dtype, acc, act=R.ACT_NONE, slope=0.2):
    """(want, bound) of an activated output from its fp64 pre-activation reference and magnitude."""
    want = _act64(pre, act, slope)
    return want, R_OUT[out_dtype] * want.abs() + L_ACT[act] * CU[acc] * mag


ACT_NAMES = ("n", "d", "h", "w", "c")
W_NAMES = ("tap", "co", "ci")


def check_output(got, pre, mag, acc, act=R.ACT_NONE, slope=0.2, what="output"):
    want, bound = output_bound(pre, mag, got.dtype, acc, act, slope)
    return check_elements(got, want, bound, what, ACT_NAMES)


def check_stats(got, pre, mag, out_dtype, acc, what="statistics"):
    """Epilogue statistics [n][c][{sum, sum of squares}] of the pre-activation output, each checked on its own."""
    got = _d(got)
    bound = R_OUT[out_dtype] * pre.abs() + CU[acc] * mag
    dims = (1, 2, 3)
    s1, b1 = pre.sum(dims), bound.sum(dims)
    s2, b2 = (pre * pre).sum(dims), ((2 * pre.abs() + bound) * bound).sum(dims)
    r1 = check_elements(got[..., 0], s1, b1, what + " sum", ("n", "c"))
    r2 = check_elements(got[..., 1], s2, b2, what + " sum of squares", ("n", "c"))
    return max(r1, r2)


def check_fprop(got_y, x, w, bias, g, acc, act=R.ACT_NONE, slope=0.2, got_stats=None, what="fprop"):
    pre, mag = fprop_ref(x, w, bias, g)
    r = check_output(got_y, pre, mag, acc, act, slope, what)
    if got_stats is not None:
        r = max(r, check_stats(got_stats, pre, mag, got_y.dtype, acc, what + " statistics"))
    return r


def check_dgrad(got_dx, dy, wT, g, acc, what="dgrad"):
    ref, mag = dgrad_ref(dy, wT, g, tuple(got_dx.shape[1:4]))
    return check_output(got_dx, ref, mag, acc, what=what)


def check_wgrad_elements(got_dw, want, mag, acc, what="wgrad"):
    return check_elements(got_dw, want, CU[acc] * mag, what, W_NAMES)


def check_dbias(got_db, dy, what="dbias", base=None):
    dy = _d(dy)
    want = dy.sum((0, 1, 2, 3)) + (0 if base is None else _d(base))
    bound = CU["fma"] * dy.abs().sum((0, 1, 2, 3)) + (0 if base is None else 2.0 ** -23 * _d(base).abs())
    return check_elements(got_db, want, bound, what, ("c",))


def check_wgrad(got_dw, x, dy, g, acc, got_db=None, base_dw=None, base_db=None, what="wgrad"):
    """dw (fp32) element by element, plus dbias; with ``base_*`` the kernel added into buffers that held these."""
    dw, mag = wgrad_ref(x, dy, g)
    bound = CU[acc] * mag
    if base_dw is not None:                # plus the fp32 rounding of the one add into the caller's buffer
        dw = dw + _d(base_dw)
        bound = bound + 2.0 ** -23 * _d(base_dw).abs()
    r = check_elements(got_dw, dw, bound, what, W_NAMES)
    if got_db is not None:
        r = max(r, check_dbias(got_db, dy, what + " dbias", base_db))
    return r
