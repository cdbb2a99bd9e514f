"""Every case of the tensor-core envelope sweep (test_conv_envelope_gpu.py) can be planned on the host: the dispatcher
routes it as expected, the implicit-GEMM plans and the persistent schedules of its three ops build (mra_conv_plan_describe,
mra_debug_schedule walk the code the kernels run), and the expected wgrad schedule shape (shared items, CTA pairs) holds.
No case that the eligibility predicates accept may be rejected later by a host-side "does not fit" / "too many taps"."""
import ctypes as C

import pytest

from mra_gan_b200 import _lib, ops
from test_conv_envelope_gpu import CASES, LOWERING, cid, desc, wgrad_schedule


@pytest.mark.parametrize("c", CASES, ids=cid)
def test_envelope_case_is_planned(c, monkeypatch):
    L = _lib.lib()
    d = desc(c)
    tcore = c.kernel != "fp32"
    for which in range(3):
        assert bool(L.mra_conv3d_uses_tensor_cores(C.byref(d), which)) == (tcore and which not in c.cc)
    assert int(L.mra_conv3d_lowering(C.byref(d))) == LOWERING[c.kernel]
    if c.kernel in ("stem", "head", "im2col", "convT1"):
        assert all(int(L.mra_conv3d_workspace_size(C.byref(d), w)) > 0 for w in range(3))
        return
    if not tcore:
        return
    for which in range(3):
        assert ops.plan_describe(c.g, c.n, c.dims, which)
        assert ops.schedule_describe(c.g, c.n, c.dims, which)
    if c.pair_min0:
        monkeypatch.setenv("MRA_WGRAD_PAIR_MIN", "0")
    pair, shared = wgrad_schedule(c)
    assert pair or not c.pair_min0
    assert c.shared is None or shared == c.shared
