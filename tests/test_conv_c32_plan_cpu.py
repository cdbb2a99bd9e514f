"""Host-side planning of the convolutions whose channel counts are multiples of 32 but not of 64 (the cases of
test_conv_c32_gpu.py): the dispatcher sends them to the tensor cores, their plans and wgrad schedules build, every
output position is produced by exactly one gather launch, the stream-K segments of the wgrad launch tile every work item's
K range exactly once and its N tiles cover [0, Cn) with the last one starting inside it.  Channel counts that are not
multiples of 32 stay on the CUDA cores, and the halo, phase and split-K kernels keep declining 32-channel shapes."""
import ctypes as C
import itertools

import pytest
import torch

from mra_gan_b200 import _lib, ops
from mra_gan_b200.ops import ConvGeom as G
from test_conv_c32_gpu import CASES
from test_conv_envelope_gpu import LOWERING, Case, cid, desc


def _gather_launches(words):
    """(o0, ostep, dims) per launch of a gather plan (layout: conv_plan.h describe())"""
    assert words[0] == 0
    p, out = 11, []
    for _ in range(words[10]):
        o0, ostep, dims = words[p:p + 3], words[p + 3], words[p + 4:p + 7]
        ntaps = words[p + 11]
        p += 12 + 4 * ntaps
        out.append((o0, ostep, dims))
    assert p == len(words)
    return out


@pytest.mark.parametrize("c", CASES, ids=cid)
def test_c32_case_is_planned(c):
    L = _lib.lib()
    d = desc(c)
    for which in range(3):
        assert bool(L.mra_conv3d_uses_tensor_cores(C.byref(d), which)) == (which not in c.cc)
    assert int(L.mra_conv3d_lowering(C.byref(d))) == LOWERING[c.kernel]
    if c.kernel != "gather":
        assert all(int(L.mra_conv3d_workspace_size(C.byref(d), w)) > 0 for w in range(3))
        return
    for which in range(2):
        if which in c.cc:
            continue
        words = ops.plan_describe(c.g, c.n, c.dims, which)
        odims = words[7:10]
        seen = {}
        for o0, ostep, dims in _gather_launches(words):
            for pos in itertools.product(*[range(o0[i], o0[i] + ostep * dims[i], ostep) for i in range(3)]):
                seen[pos] = seen.get(pos, 0) + 1
        assert set(seen) == set(itertools.product(*[range(o) for o in odims])), "output positions not covered"
        assert all(v == 1 for v in seen.values()), "an output position produced twice"
        # no halo-plane launch (they need multiples of 64): the per-tap kernel takes every launch
        assert ops.schedule_describe(c.g, c.n, c.dims, which)[1] == 0
    assert ops.plan_describe(c.g, c.n, c.dims, 2)
    w = ops.schedule_describe(c.g, c.n, c.dims, 2)
    pair, m_tiles, n_tiles, n_groups, n_items, kblocks = w[1], w[2], w[3], w[4], w[5], w[6]
    assert pair == 0
    g = c.g
    km, kn = (g.cin, g.cout) if g.transposed else (g.cout, g.cin)      # dense (M) / shifted (N) operand channels
    ncc = 4 if kn % 256 == 0 else (2 if kn % 128 == 0 else 1)          # 64-channel chunks of the shifted operand per tap
    assert (m_tiles - 1) * 128 < km <= m_tiles * 128
    assert (n_tiles - 1) * 64 * ncc < kn <= n_tiles * 64 * ncc
    at = 10 + 5 * n_groups
    segs = [w[at + 1 + 9 * i: at + 10 + 9 * i] for i in range(w[at])]
    cover = {}
    for (u, item, mt, nt, grp, tap0, ntap, kb0, kb1) in segs:
        assert 0 <= mt < m_tiles and 0 <= nt < n_tiles and 0 <= item < n_items and 0 <= kb0 < kb1 <= kblocks
        cover.setdefault((item, mt, nt), []).append((kb0, kb1))
    assert len(cover) == n_items * m_tiles * n_tiles
    for ranges in cover.values():
        ranges.sort()
        assert ranges[0][0] == 0 and ranges[-1][1] == kblocks
        assert all(a[1] == b[0] for a, b in zip(ranges, ranges[1:])), "K range of a work item not tiled exactly once"


@pytest.mark.parametrize("cin,cout", [(8, 64), (64, 16), (24, 24), (40, 64), (64, 48), (48, 96), (1, 16), (24, 1)])
def test_channels_not_multiples_of_32_stay_on_the_cuda_cores(cin, cout):
    I = ops.CudaImpl()
    for k, s in ((3, 1), (4, 2), (7, 1)):
        g = G(cin, cout, k, s, 0)
        for which in range(3):
            assert not I.conv_uses_tensor_cores(g, 1, (16, 16, 16), torch.bfloat16, which)


@pytest.mark.parametrize("g,dims", [(G(64, 32, 3, 2, 1, True, 1), (8, 8, 8)), (G(32, 64, 4, 2, 1), (16, 16, 16)),
                                    (G(32, 32, 4, 2, 1), (2, 2, 2))])
def test_phase_and_split_k_decline_32_multiples(g, dims, monkeypatch):
    """the opt-in phase-halo kernel and split-K need multiples of 64: no split-K workspace is asked for, and with the
    phase kernel switched on the plan still has no halo-plane launch"""
    L = _lib.lib()
    d = desc(Case("gather", g, dims, 1))
    for which in range(2):
        assert int(L.mra_conv3d_workspace_size(C.byref(d), which)) == 0
    monkeypatch.setenv("MRA_GATHER_PHASE", "1")
    for which in range(2):
        assert ops.schedule_describe(g, 1, dims, which)[1] == 0
