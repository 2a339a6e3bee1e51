"""Head dims above 128 on the exact (fp32 FFMA) route without a device: the workspace covers the per-chunk states for
every DHQK <= 256, DHHV <= 512 (multiples of 4) in fp32 and, with impl = EXACT, in 16-bit; pairs past those limits keep
the 256-byte "unsupported" size; and the chunkwise custom-op fakes at fp32 (256, 512) report no c_states."""
import ctypes
import os
import sys

import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import __graft_entry__ as G  # noqa: E402

ops = torch.ops.mlstm_b200
PAIRS = [(256, 512), (256, 256), (128, 256), (128, 512), (132, 260)]


@pytest.fixture(scope="module")
def pkg():
    G.build()
    import xlstm_yolo_clean_b200 as p

    return p


def _workspace(pkg, DK, DV, dtype, impl, backward, B=2, NH=3, S=512, chunk=64):
    s = pkg._cabi.Shape()
    s.B, s.NH, s.S, s.DHQK, s.DHHV, s.chunk_size, s.dtype, s.impl = B, NH, S, DK, DV, chunk, dtype, impl
    return pkg.load_library().mlstm_b200_workspace_bytes(ctypes.byref(s), backward)


@pytest.mark.parametrize("DK,DV", PAIRS)
def test_workspace_holds_the_chunk_states(pkg, DK, DV):
    """The states entering every internal chunk and the final one, (S / L + 1) of them with L <= 64, are DHQK x DHHV
    fp32 each; the backward holds their gradients as well."""
    C = pkg._cabi
    B, NH, S = 2, 3, 512
    per_state = B * NH * DK * DV * 4
    for dtype, impl in ((C.F32, C.IMPL_AUTO), (C.F32, C.IMPL_EXACT), (C.BF16, C.IMPL_EXACT), (C.F16, C.IMPL_EXACT)):
        fw = _workspace(pkg, DK, DV, dtype, impl, 0, B, NH, S)
        bw = _workspace(pkg, DK, DV, dtype, impl, 1, B, NH, S)
        assert fw >= (S // 64 + 1) * per_state, (dtype, impl, fw)
        assert bw >= 2 * (S // 64 + 1) * per_state, (dtype, impl, bw)
    for chunk in (16, 64):  # S = chunk: one chunk, two states
        assert _workspace(pkg, DK, DV, C.F32, C.IMPL_AUTO, 1, B, NH, chunk, chunk) >= 2 * 2 * per_state


@pytest.mark.parametrize("DK,DV", [(260, 512), (512, 512), (256, 516), (254, 512)])
def test_pairs_past_the_limits_stay_unsupported(pkg, DK, DV):
    C = pkg._cabi
    for backward in (0, 1):
        for dtype in (C.F32, C.BF16):
            assert _workspace(pkg, DK, DV, dtype, C.IMPL_EXACT, backward) == 256


def test_fp32_wide_fakes_report_no_c_states(pkg):
    DK, DV = 256, 512
    B, NH, S = 2, 3, 256
    with FakeTensorMode():
        mk = lambda *s: torch.empty(*s, device="cuda", dtype=torch.float32)  # noqa: E731
        q, k, v, i, f = mk(B, NH, S, DK), mk(B, NH, S, DK), mk(B, NH, S, DV), mk(B, NH, S), mk(B, NH, S)
        h, nm, cl, nl, ml, cs = ops.chunkwise_fw(q, k, v, i, f, None, None, None, None, None, True, 64, 1e-6, 0, True,
                                                 False, False, 0.0, None)
        assert h.shape == (B, NH, S, DV) and h.dtype == torch.float32
        assert cl.shape == (B, NH, DK, DV) and nl.shape == (B, NH, DK) and ml.shape == (B, NH, 1)
        assert cs.numel() == 0
        grads = ops.chunkwise_bw(q, k, v, i, f, nm[0], nm[1], h, None, None, None, None, cs, None, None, 64, 1e-6, 0,
                                 False, False, False, 0.0, None)
        for g, shp in zip(grads, ((B, NH, S, DK), (B, NH, S, DK), (B, NH, S, DV), (B, NH, S), (B, NH, S))):
            assert g.shape == shp and g.dtype == torch.float32
