"""The ``mlstm_b200`` custom ops (xlstm_yolo_clean_b200/ops.py) without a device: fake (meta) implementations on fake
CUDA tensors allocate exactly what the real ones do -- shapes, dtypes, strides, the c_states size the C-ABI reports --
a symbolic batch size traces, and eager calls never enter the ops."""
import ctypes as C
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
HEAD_DIMS = [(32, 32), (64, 64), (128, 128), (32, 64), (64, 128)]
F32, U8 = torch.float32, torch.uint8


@pytest.fixture(scope="module")
def pkg():
    G.build()
    import xlstm_yolo_clean_b200 as p

    return p


def _contig(*shape):
    st, acc = [], 1
    for s in reversed(shape):
        st.append(acc)
        acc *= s
    return tuple(reversed(st))


def _check(t, shape, dtype):
    assert tuple(t.shape) == tuple(shape) and t.dtype == dtype and t.stride() == _contig(*shape), (t.shape, t.dtype, t.stride())
    assert t.device.type == "cuda"


def _states_bytes(pkg, B, NH, S, DK, DV, dtype, chunk=64):
    s = pkg._cabi.Shape()
    s.B, s.NH, s.S, s.DHQK, s.DHHV, s.chunk_size = B, NH, S, DK, DV, chunk
    s.dtype, s.impl = pkg.backend._DTYPES[dtype], pkg._cabi.IMPL_AUTO
    return pkg.load_library().mlstm_b200_states_bytes(C.byref(s))


def _heads(B, NH, S, DK, DV, dtype):
    mk = lambda *s: torch.empty(*s, device="cuda", dtype=dtype)  # noqa: E731
    return mk(B, NH, S, DK), mk(B, NH, S, DK), mk(B, NH, S, DV), mk(B, NH, S), mk(B, NH, S)


CASES = [(dk, dv, torch.bfloat16) for dk, dv in HEAD_DIMS] + [(64, 64, torch.float32)]  # the last: exact (FFMA) route


@pytest.mark.parametrize("DK,DV,dtype", CASES)
def test_chunkwise_fakes(pkg, DK, DV, dtype):
    B, NH, S = 3, 2, 320
    with FakeTensorMode():
        q, k, v, i, f = _heads(B, NH, S, DK, DV, dtype)
        c0 = torch.empty(B, NH, DK, DV, device="cuda")
        for save, last in ((True, True), (False, False)):
            h, nm, cl, nl, ml, cs = ops.chunkwise_fw(q, k, v, i, f, c0, None, None, None, None, last, 64, 1e-6, 0, save, False,
                                                     False, 0.0, None)
            _check(h, (B, NH, S, DV), dtype)
            _check(nm, (2, B, NH, S), F32)
            if last:
                _check(cl, (B, NH, DK, DV), F32), _check(nl, (B, NH, DK), F32), _check(ml, (B, NH, 1), F32)
            else:
                assert cl.numel() == nl.numel() == ml.numel() == 0
            want = _states_bytes(pkg, B, NH, S, DK, DV, dtype) if save else 0
            assert cs.dtype == U8 and cs.numel() == want
            assert (want > 0) == (save and dtype != F32)  # the exact route recomputes its states
        grads = ops.chunkwise_bw(q, k, v, i, f, nm[0], nm[1], h, c0, None, None, None, cs, None, None, 64, 1e-6, 0, True,
                                 False, False, 0.0, torch.float16)
        gdt = torch.float16 if dtype != F32 else F32  # the exact route writes its own dtype
        for g, shp in zip(grads, ((B, NH, S, DK), (B, NH, S, DK), (B, NH, S, DV), (B, NH, S), (B, NH, S))):
            _check(g, shp, gdt)
        _check(grads[5], (B, NH, DK, DV), F32)
        # the custom_fwd rule: fp16 inputs rounded to the bf16 kernel dtype inside the op
        q16, k16, v16, i16, f16 = _heads(B, NH, S, DK, DV, torch.float16)
        h = ops.chunkwise_fw(q16, k16, v16, i16, f16, None, None, None, torch.bfloat16, None, False, 64, 1e-6, 0, True, False,
                             False, 0.0, None)[0]
        _check(h, (B, NH, S, DV), torch.bfloat16)


@pytest.mark.parametrize("DK,DV", HEAD_DIMS)
def test_layer_and_epilogue_fakes(pkg, DK, DV):
    B, NH, S = 2, 4, 400
    H = NH * DV
    with FakeTensorMode():
        qk = torch.empty(B, S, 2 * NH * DK, device="cuda", dtype=torch.float16)
        v = torch.empty(B, S, H, device="cuda", dtype=torch.float16)
        gates = torch.empty(B, S, 2 * NH, device="cuda", dtype=torch.float16)
        h, nm, cs = ops.layer_fw(qk, v, gates, NH, torch.bfloat16, 16, 1e-6, 0, True, False, False, 15.0, torch.float16)
        _check(h, (B, NH, S, DV), torch.bfloat16)
        _check(nm, (2, B, NH, S), F32)
        assert cs.numel() == _states_bytes(pkg, B, NH, S, DK, DV, torch.bfloat16, 16) > 0
        d_qk, d_v, d_g = ops.layer_bw(qk, v, gates, nm, h, cs, NH, torch.bfloat16, 16, 1e-6, 0, False, False, 15.0,
                                      torch.float16)
        _check(d_qk, qk.shape, torch.float16), _check(d_v, v.shape, torch.float16), _check(d_g, gates.shape, torch.float16)
        w = torch.empty(H, device="cuda")
        xs = torch.empty(B, S, H, device="cuda", dtype=torch.float16)
        for save in (True, False):
            y, h, nm, cs = ops.chunkwise_fw_epilogue(qk, v, gates, xs, w, w, w, NH, torch.bfloat16, 16, 1e-6, 0, save, True,
                                                     False, 15.0, 1e-6, torch.float16, torch.float16)
            _check(y, (B, S, H), torch.float16)
            _check(nm, (2, B, NH, S), F32)
            if save:
                _check(h, (B, NH, S, DV), torch.bfloat16)
            assert h.numel() == (h.numel() if save else 0) and (cs.numel() > 0) == save


def test_cellout_rmsnorm_convert_recurrent_fakes(pkg):
    B, NH, S, D = 2, 4, 77, 64
    with FakeTensorMode():
        big = torch.empty(B, NH, S + 3, D, device="cuda", dtype=torch.bfloat16)
        h = big[:, :, 3:]  # a strided h: dh takes its strides
        w = torch.empty(NH * D, device="cuda")
        x = torch.empty(B, S, NH * D, device="cuda", dtype=torch.float16)
        _check(ops.cellout_fw(h, w, w, w, x, 1e-6, torch.float16), (B, S, NH * D), torch.float16)
        dh, dpar, dx = ops.cellout_bw(h, x, w, w, x, 1e-6, torch.float16, True)
        assert dh.shape == h.shape and dh.stride() == h.stride() and dh.dtype == h.dtype
        _check(dpar, (3, NH * D), F32), _check(dx, (B, S, NH * D), torch.float16)
        assert ops.cellout_bw(h, None, w, None, x, 1e-6, torch.float16, True)[2].numel() == 0
        x2 = torch.empty(B * S, 256, device="cuda", dtype=torch.float32)
        y, rstd = ops.rmsnorm_fw(x2, w[:256], 1e-6, torch.float16)
        _check(y, (B * S, 256), torch.float16), _check(rstd, (B * S,), F32)
        dx, dw = ops.rmsnorm_bw(x2, w[:256], rstd, y, 1e-6, torch.float16)
        _check(dx, (B * S, 256), F32), _check(dw, (256,), F32)
        perm = torch.empty(B, S, NH, D, device="cuda", dtype=torch.float16).transpose(1, 2)  # dense, permuted
        c = ops.convert16(perm, torch.bfloat16)
        assert c.dtype == torch.bfloat16 and c.stride() == perm.stride()
        q, k, v, i, f = _heads(B, NH, 16, 64, 128, torch.bfloat16)
        hr, cl, nl, ml = ops.recurrent_sequence(q, k, v, i, f, None, None, None, True, 1e-6, False)
        _check(hr, (B, NH, 16, 128), torch.bfloat16)
        _check(cl, (B, NH, 64, 128), F32), _check(nl, (B, NH, 64), F32), _check(ml, (B, NH, 1), F32)


def test_export_with_symbolic_batch(pkg):
    """torch.export of the drop-in call with the batch dimension symbolic."""

    class M(torch.nn.Module):
        def forward(self, q, k, v, i, f):
            return pkg.mlstm_chunkwise__b200(q, k, v, i, f, chunk_size=64, return_last_states=True)

    B = torch.export.Dim("B", min=2, max=64)
    with FakeTensorMode(allow_non_fake_inputs=True):
        args = _heads(4, 2, 128, 64, 64, torch.bfloat16)
        ep = torch.export.export(M(), args, dynamic_shapes={n: {0: B} for n in ("q", "k", "v", "i", "f")})
    node = [n for n in ep.graph.nodes if n.target is ops.chunkwise_fw.default]
    assert len(node) == 1
    h, nm, c_last = node[0].meta["val"][:3]
    assert all(isinstance(t.shape[0], torch.SymInt) for t in (h, c_last)) and isinstance(nm.shape[1], torch.SymInt)


def test_states_bytes_scale_with_symbolic_batch(pkg):
    from torch._dynamo.source import ConstantSource
    from torch.fx.experimental.symbolic_shapes import ShapeEnv

    env = ShapeEnv()
    B = env.create_symintnode(env.create_symbol(5, ConstantSource("B")), hint=5)
    with FakeTensorMode(shape_env=env):
        q = torch.empty(B, 2, 128, 64, device="cuda", dtype=torch.bfloat16)
        gate = torch.empty(B, 2, 128, device="cuda", dtype=torch.bfloat16)
        cs = ops.chunkwise_fw(q, q, q, gate, gate, None, None, None, None, None, False, 64, 1e-6, 0, True, False, False, 0.0,
                              None)[5]
    assert isinstance(cs.shape[0], torch.SymInt)  # not specialised to the hint
    assert cs.shape[0] == B * _states_bytes(pkg, 1, 2, 128, 64, 64, torch.bfloat16)
    assert _states_bytes(pkg, 5, 2, 128, 64, 64, torch.bfloat16) == 5 * _states_bytes(pkg, 1, 2, 128, 64, 64, torch.bfloat16)


def test_eager_calls_never_enter_the_ops(pkg, monkeypatch):
    """Every compile-path function raises if reached: eager entry points still refuse CPU tensors their own way."""
    from xlstm_yolo_clean_b200 import ops as O

    class Entered(Exception):
        pass

    def boom(*a, **k):
        raise Entered

    for name in ("chunkwise_fw", "chunkwise_bw", "layer_fw", "layer_bw", "chunkwise_fw_epilogue", "cellout_fw", "cellout_bw",
                 "rmsnorm_fw", "rmsnorm_bw", "_convert16", "_recurrent_sequence", "chunkwise_function", "fw_launch",
                 "bw_launch", "rms_norm", "convert16", "recurrent_sequence"):
        monkeypatch.setattr(O, name, boom)
    q, k, v = (torch.randn(1, 2, 64, 32) for _ in range(3))
    i, f = torch.randn(1, 2, 64), torch.randn(1, 2, 64)
    calls = [
        lambda: pkg.mlstm_chunkwise__b200(q, k, v, i, f),
        lambda: pkg.mlstm_siging_chunkwise__b200(q, k, v, i, f),
        lambda: pkg.mlstm_chunkwise_fw(q, k, v, i, f),
        lambda: pkg.mlstm_chunkwise_bw(q, k, v, i, f, i, i, q),
        lambda: pkg.mlstm_recurrent_sequence__b200(q, k, v, i, f),
        lambda: pkg.cell_out(torch.randn(1, 2, 8, 64)),
        lambda: pkg.rms_norm_b200(torch.randn(2, 256), torch.ones(256)),
        lambda: pkg.vil._layer_layout(torch.randn(1, 64, 128), torch.randn(1, 64, 64), torch.randn(1, 64, 4), 2, False, False,
                                      64, 1e-6, torch.bfloat16, 0.0),
        lambda: pkg.vil._cell_fused(torch.randn(1, 64, 128), torch.randn(1, 64, 64), torch.randn(1, 64, 4), None, None, None,
                                    None, 2, False, False, 64, 1e-6, torch.bfloat16, 0.0, 1e-6, torch.float16),
    ]
    for call in calls:
        with pytest.raises((RuntimeError, AssertionError)) as e:
            call()
        assert not isinstance(e.value, Entered)
    assert pkg.convert16(torch.randn(4, dtype=torch.float16), torch.bfloat16).dtype == torch.bfloat16  # torch's cast on CPU
