"""xLSTM-Large's head geometry (DHQK, DHHV) = (256, 512) (qk_dim_factor 0.5 at embedding 4096, 8 heads) without a
device: the support matrix of the tensor-core route (16-bit, S % 4 == 0; its neighbours and fp32 stay where they were),
the c_states / workspace sizes, and the custom-op fakes and torch.export at this pair."""
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
DK, DV = 256, 512
F32, U8 = torch.float32, torch.uint8


@pytest.fixture(scope="module")
def pkg():
    G.build()
    import xlstm_yolo_clean_b200 as p

    return p


def _shape(pkg, DK_, DV_, dtype, S=256, B=2, NH=4, chunk=64):
    s = pkg._cabi.Shape()
    s.B, s.NH, s.S, s.DHQK, s.DHHV, s.chunk_size, s.dtype, s.impl = B, NH, S, DK_, DV_, chunk, dtype, pkg._cabi.IMPL_AUTO
    return s


def _supported(pkg, DK_, DV_, dtype, S=256):
    return bool(pkg.load_library().mlstm_b200_tensor_path_supported(ctypes.byref(_shape(pkg, DK_, DV_, dtype, S))))


def test_wide_pair_supported_in_16_bit(pkg):
    C = pkg._cabi
    for dt in (C.BF16, C.F16):
        assert _supported(pkg, DK, DV, dt)
        assert _supported(pkg, DK, DV, dt, S=196)  # ragged last tile
        assert not _supported(pkg, DK, DV, dt, S=198)  # S % 4 != 0
    assert not _supported(pkg, DK, DV, C.F32)  # the exact route stays at head dims <= 128
    for dt in (torch.bfloat16, torch.float16):
        assert pkg.tensor_path_supported(1, 8, 4096, DK, DV, dt)
    assert (DK, DV) in pkg.vil.TENSOR_HEAD_DIMS


@pytest.mark.parametrize("DK_,DV_", [(256, 256), (128, 256), (128, 512), (512, 512), (512, 256)])
def test_neighbours_stay_unsupported(pkg, DK_, DV_):
    C = pkg._cabi
    for dt in (C.BF16, C.F16, C.F32):
        assert not _supported(pkg, DK_, DV_, dt)


def test_wide_state_and_workspace_sizes(pkg):
    """c_states: one 16-bit 256 x 512 state per (batch, head, 128-token tile); the backward's workspace covers the 4 x 8
    block problems; the fp32 (exact) route saves no states."""
    lib, C = pkg.load_library(), pkg._cabi
    for B, NH, S in ((2, 3, 196), (1, 8, 4096)):
        s = _shape(pkg, DK, DV, C.BF16, S, B, NH, chunk=4)
        NT = (S + 127) // 128
        assert lib.mlstm_b200_states_bytes(ctypes.byref(s)) == B * NH * NT * DK * DV * 2
        assert lib.mlstm_b200_workspace_bytes(ctypes.byref(s), 1) > 0
    assert lib.mlstm_b200_states_bytes(ctypes.byref(_shape(pkg, DK, DV, C.F32))) == 0


def _contig(*shape):
    st, acc = [], 1
    for s in reversed(shape):
        st.append(acc)
        acc *= s
    return tuple(reversed(st))


def _check(t, shape, dtype):
    assert tuple(t.shape) == tuple(shape) and t.dtype == dtype and t.stride() == _contig(*shape), (t.shape, t.dtype, t.stride())


def _states_bytes(pkg, B, NH, S, dtype, chunk=64):
    s = _shape(pkg, DK, DV, pkg.backend._DTYPES[dtype], S, B, NH, chunk)
    return pkg.load_library().mlstm_b200_states_bytes(ctypes.byref(s))


def _heads(B, NH, S, dtype):
    mk = lambda *s: torch.empty(*s, device="cuda", dtype=dtype)  # noqa: E731
    return mk(B, NH, S, DK), mk(B, NH, S, DK), mk(B, NH, S, DV), mk(B, NH, S), mk(B, NH, S)


def test_chunkwise_and_layer_fakes(pkg):
    B, NH, S = 3, 2, 320
    with FakeTensorMode():
        q, k, v, i, f = _heads(B, NH, S, torch.bfloat16)
        c0 = torch.empty(B, NH, DK, DV, device="cuda")
        for save, last in ((True, True), (False, False)):
            h, nm, cl, nl, ml, cs = ops.chunkwise_fw(q, k, v, i, f, c0, None, None, None, None, last, 64, 1e-6, 0, save, False,
                                                     False, 0.0, None)
            _check(h, (B, NH, S, DV), torch.bfloat16)
            _check(nm, (2, B, NH, S), F32)
            if last:
                _check(cl, (B, NH, DK, DV), F32), _check(nl, (B, NH, DK), F32), _check(ml, (B, NH, 1), F32)
            assert cs.dtype == U8 and cs.numel() == (_states_bytes(pkg, B, NH, S, torch.bfloat16) if save else 0)
        assert cs.numel() == 0 and _states_bytes(pkg, B, NH, S, torch.bfloat16) == B * NH * 3 * DK * DV * 2
        _, nm, _, _, _, cs = ops.chunkwise_fw(q, k, v, i, f, None, None, None, None, None, False, 64, 1e-6, 0, True, False,
                                              False, 0.0, None)
        grads = ops.chunkwise_bw(q, k, v, i, f, nm[0], nm[1], h, c0, None, None, None, cs, None, None, 64, 1e-6, 0, True,
                                 False, False, 0.0, torch.float16)
        for g, shp in zip(grads, ((B, NH, S, DK), (B, NH, S, DK), (B, NH, S, DV), (B, NH, S), (B, NH, S))):
            _check(g, shp, torch.float16)
        _check(grads[5], (B, NH, DK, DV), F32)
        # layer layout (B, S, NH * D): xLSTM-Large's projections
        qk = torch.empty(B, S, 2 * NH * DK, device="cuda", dtype=torch.float16)
        vl = torch.empty(B, S, NH * DV, device="cuda", dtype=torch.float16)
        gates = torch.empty(B, S, 2 * NH, device="cuda", dtype=torch.float16)
        h, nm, cs = ops.layer_fw(qk, vl, gates, NH, torch.bfloat16, 16, 1e-6, 0, True, False, False, 15.0, torch.float16)
        _check(h, (B, NH, S, DV), torch.bfloat16)
        assert cs.numel() == _states_bytes(pkg, B, NH, S, torch.bfloat16, 16) > 0
        d_qk, d_v, d_g = ops.layer_bw(qk, vl, gates, nm, h, cs, NH, torch.bfloat16, 16, 1e-6, 0, False, False, 15.0,
                                      torch.float16)
        _check(d_qk, qk.shape, torch.float16), _check(d_v, vl.shape, torch.float16), _check(d_g, gates.shape, torch.float16)
        hr, cl, nl, ml = ops.recurrent_sequence(q, k, v, i, f, None, None, None, True, 1e-6, False)
        _check(hr, (B, NH, S, DV), torch.bfloat16)
        _check(cl, (B, NH, DK, DV), F32), _check(nl, (B, NH, DK), F32), _check(ml, (B, NH, 1), F32)


def test_export_with_symbolic_batch(pkg):
    """torch.export of the drop-in call at (256, 512) with the batch dimension symbolic: the c_states size is traced as
    a multiple of B."""

    class M(torch.nn.Module):
        def forward(self, q, k, v, i, f):
            return pkg.mlstm_chunkwise__b200(q, k, v, i, f, chunk_size=64, return_last_states=True)

    B = torch.export.Dim("B", min=2, max=64)
    with FakeTensorMode(allow_non_fake_inputs=True):
        args = _heads(4, 2, 256, torch.bfloat16)
        ep = torch.export.export(M(), args, dynamic_shapes={n: {0: B} for n in ("q", "k", "v", "i", "f")})
    node = [n for n in ep.graph.nodes if n.target is ops.chunkwise_fw.default]
    assert len(node) == 1
    h, nm, c_last = node[0].meta["val"][:3]
    assert all(isinstance(t.shape[0], torch.SymInt) for t in (h, c_last)) and isinstance(nm.shape[1], torch.SymInt)
    assert tuple(h.shape[1:]) == (2, 256, DV) and tuple(c_last.shape[1:]) == (2, DK, DV)
