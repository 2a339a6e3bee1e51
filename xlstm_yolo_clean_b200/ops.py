"""The C-ABI calls as ``torch.library`` custom ops (namespace ``mlstm_b200``), so that ``torch.compile`` and
``torch.export`` trace the B200 kernels as opaque graph nodes instead of breaking the graph at every ctypes call.

Dynamo cannot trace what the eager entry points do around a launch (ctypes, ``data_ptr()`` arithmetic, the per-thread
call plans), so while it traces (``torch.compiler.is_compiling()``) those entry points call these ops instead of their
``autograd.Function``s, after the same host decisions -- chunk size, padding, one launch or two, gradient dtype -- made by
the same functions, in Python, where Dynamo guards on them; the decisions depend on sizes, strides and dtypes only.
Eager calls never come here.

Each op's real implementation is the body the eager ``autograd.Function`` calls (``backend._fw_launch`` /
``_chunkwise_bw``, ``vil._layer_fw`` / ``_layer_bw`` / ``_cell_fused_fw``, ``vil._cellout_fw_call`` / ``_cellout_bw_call``,
``vil._rmsnorm_fw_call`` / ``_rmsnorm_bw_call``), so it runs exactly the kernels an eager call runs.  Each fake
implementation allocates exactly what the real one does, shapes, dtypes and strides, and takes a symbolic batch size.
An op cannot return None: absent outputs are 0-element tensors, mapped back to None by the few wrappers here.  No output
aliases an input.

Inputs the eager ``autograd.Function``s round to the kernel dtype inside their forward (``custom_fwd(cast_inputs=...)``,
``convert16`` of the layer tensors) are rounded inside the ops too, so the gradients reach the caller's tensors through
one cast, as in eager mode.  The backward ops round the saved caller tensors again instead of keeping the rounded
copies alive (under autocast: one conversion pass per input and backward).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch
from torch import Tensor

from . import _cabi
from . import backend as _backend
from . import vil as _vil

_F32, _U8 = torch.float32, torch.uint8
# Inductor hands each op exactly the strides its fake saw: dh of the cell-output backward takes h's strides
_TAGS = (torch._C.Tag.needs_exact_strides,)


def _op(name):
    return torch.library.custom_op(f"mlstm_b200::{name}", mutates_args=(), tags=_TAGS)


def _none(t: Optional[Tensor]) -> Optional[Tensor]:
    return None if t is None or t.numel() == 0 else t


def _empty(ref: Tensor, dtype=_F32) -> Tensor:
    return ref.new_empty(0, dtype=dtype)


def _autocast_eligible(t: Optional[Tensor]) -> bool:
    """What custom_fwd(cast_inputs=...) re-rounds: floating CUDA tensors other than float64."""
    return t is not None and t.is_floating_point() and t.is_cuda and t.dtype is not torch.float64


def _cast(dtype: Optional[torch.dtype], *ts):
    if dtype is None:
        return ts
    return tuple(t.to(dtype) if _autocast_eligible(t) else t for t in ts)


def _shape_struct(NH, S, DK, DV, dtype, chunk_size, impl) -> _cabi.Shape:
    """The C-ABI shape with B = 1: what the host-only queries read does not depend on B (states scale with it)."""
    s = _cabi.Shape()
    s.B, s.NH, s.S, s.DHQK, s.DHHV = 1, int(NH), int(S), int(DK), int(DV)
    s.chunk_size, s.dtype, s.impl = int(chunk_size), _backend._DTYPES[dtype], int(impl)
    return s


def _tensor_route(NH, S, DK, DV, dtype, chunk_size, impl) -> bool:
    return _backend._tensor_route(_cabi.load_library(), _shape_struct(NH, S, DK, DV, dtype, chunk_size, impl))


def _states_bytes(B, NH, S, DK, DV, dtype, chunk_size, impl):
    """Size of c_states (``mlstm_b200_states_bytes``, a host-only query): linear in B, which may be symbolic."""
    return B * _cabi.load_library().mlstm_b200_states_bytes(C.byref(_shape_struct(NH, S, DK, DV, dtype, chunk_size, impl)))


# ------------------------------------------------------------------------------------------------------------------
# chunkwise mLSTM on (B, NH, S, D) tensors: mlstm_chunkwise__b200 / _siging_ and mlstm_chunkwise_fw / _bw
# ------------------------------------------------------------------------------------------------------------------
@_op("chunkwise_fw")
def chunkwise_fw(q: Tensor, k: Tensor, v: Tensor, i: Tensor, f: Tensor, c_initial: Optional[Tensor],
                 n_initial: Optional[Tensor], m_initial: Optional[Tensor], cast_to: Optional[torch.dtype],
                 qk_scale: Optional[float], return_last_states: bool, chunk_size: int, eps: float, impl: int,
                 save_states: bool, reverse: bool, siging: bool, soft_cap: float, grad_dtype: Optional[torch.dtype],
                 normalize: bool = True) -> tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """Returns h, nm = [n_out, m_out] (2, B, NH, S) fp32, C / n / m_last fp32 (0-element unless
    ``return_last_states``), c_states uint8 (0-element unless saved).  ``cast_to``: the custom_fwd rule, every floating
    input rounded to that dtype first.  ``grad_dtype`` is read by the backward only.  ``normalize=False``: the
    sigmoid-input-gate variant without the normaliser (``siging`` must be set)."""
    mode = _backend._siging_mode(siging, normalize)
    q, k, v, i, f, c0, n0, m0 = _cast(cast_to, q, k, v, i, f, c_initial, n_initial, m_initial)
    h, nm, last, c_states = _backend._fw_launch(q, k, v, i, f, c0, n0, m0, qk_scale, return_last_states, chunk_size, eps,
                                                impl, save_states, reverse, mode, soft_cap)
    last = last if last is not None else tuple(_empty(q) for _ in range(3))
    return h, nm, *last, (c_states if c_states is not None else _empty(q, _U8))


@chunkwise_fw.register_fake
def _(q, k, v, i, f, c_initial, n_initial, m_initial, cast_to, qk_scale, return_last_states, chunk_size, eps, impl,
      save_states, reverse, siging, soft_cap, grad_dtype, normalize=True):
    _backend._siging_mode(siging, normalize)
    dt = cast_to or q.dtype
    B, NH, S, DK = q.shape
    DV = v.shape[3]
    h = q.new_empty((B, NH, S, DV), dtype=dt)
    nm = q.new_empty((2, B, NH, S), dtype=_F32)
    if return_last_states:
        last = (q.new_empty((B, NH, DK, DV), dtype=_F32), q.new_empty((B, NH, DK), dtype=_F32),
                q.new_empty((B, NH, 1), dtype=_F32))
    else:
        last = tuple(_empty(q) for _ in range(3))
    nbytes = _states_bytes(B, NH, S, DK, DV, dt, chunk_size, impl) if save_states else 0
    return h, nm, *last, q.new_empty(nbytes, dtype=_U8)


@_op("chunkwise_bw")
def chunkwise_bw(q: Tensor, k: Tensor, v: Tensor, i: Tensor, f: Tensor, n_out: Tensor, m_out: Tensor, dh: Tensor,
                 c_initial: Optional[Tensor], n_initial: Optional[Tensor], m_initial: Optional[Tensor],
                 dc_last: Optional[Tensor], c_states: Optional[Tensor], cast_to: Optional[torch.dtype],
                 qk_scale: Optional[float], chunk_size: int, eps: float, impl: int, want_dc_initial: bool, reverse: bool,
                 siging: bool, soft_cap: float, grad_dtype: Optional[torch.dtype], normalize: bool = True
                 ) -> tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """Returns dq, dk, dv, di, df (in ``grad_dtype`` where the kernels write it, else the kernel dtype) and dC_initial
    fp32 (0-element unless ``want_dc_initial``).  A 0-element ``c_states``: the kernels recompute the states."""
    mode = _backend._siging_mode(siging, normalize)
    q, k, v, i, f, c0, n0, m0 = _cast(cast_to, q, k, v, i, f, c_initial, n_initial, m_initial)
    dq, dk, dv, di, df, dc0 = _backend._chunkwise_bw(q, k, v, i, f, n_out, m_out, dh, c0, n0, m0, dc_last, qk_scale,
                                                     chunk_size, eps, impl, want_dc_initial, _none(c_states), reverse, mode,
                                                     None, soft_cap, grad_dtype)
    return dq, dk, dv, di, df, (dc0 if dc0 is not None else _empty(q))


@chunkwise_bw.register_fake
def _(q, k, v, i, f, n_out, m_out, dh, c_initial, n_initial, m_initial, dc_last, c_states, cast_to, qk_scale, chunk_size,
      eps, impl, want_dc_initial, reverse, siging, soft_cap, grad_dtype, normalize=True):
    _backend._siging_mode(siging, normalize)
    B, NH, S, DK = q.shape
    DV = v.shape[3]
    dt = cast_to or q.dtype
    route = grad_dtype not in (None, dt) and _tensor_route(NH, S, DK, DV, dt, chunk_size, impl)  # asked only when it matters
    gdt = _backend._grad_dtype(dt, grad_dtype, route)
    dc0 = q.new_empty((B, NH, DK, DV), dtype=_F32) if want_dc_initial else _empty(q)
    return (q.new_empty((B, NH, S, DK), dtype=gdt), q.new_empty((B, NH, S, DK), dtype=gdt),
            q.new_empty((B, NH, S, DV), dtype=gdt), q.new_empty((B, NH, S), dtype=gdt), q.new_empty((B, NH, S), dtype=gdt),
            dc0)


def _chunkwise_setup(ctx, inputs, output):
    (q, k, v, i, f, c0, n0, m0, cast_to, qk_scale, rls, chunk_size, eps, impl, save_states, reverse, siging, soft_cap,
     grad_dtype, normalize) = inputs
    ctx.save_for_backward(q, k, v, i, f, c0, n0, m0, output[1], output[5])
    ctx.cfg = (cast_to, qk_scale, rls, chunk_size, eps, impl, reverse, siging, soft_cap, grad_dtype, normalize)
    ctx.set_materialize_grads(False)  # nm and c_states carry no gradient: no zero tensors for them


def _chunkwise_backward(ctx, dh, dnm, dc_last, dn_last, dm_last, dc_states):
    q, k, v, i, f, c0, n0, m0, nm, c_states = ctx.saved_tensors
    cast_to, qk_scale, rls, chunk_size, eps, impl, reverse, siging, soft_cap, grad_dtype, normalize = ctx.cfg
    B, NH, S, DK = q.shape
    DV = v.shape[3]
    if dh is None:
        dh = q.new_zeros((B, NH, S, DV), dtype=cast_to or q.dtype)
    if not rls:
        dc_last = None
    elif dc_last is None:  # an unused C_last: the zeros eager autograd materialises
        dc_last = q.new_zeros((B, NH, DK, DV), dtype=_F32)
    dq, dk, dv, di, df, dc0 = chunkwise_bw(q, k, v, i, f, nm[0], nm[1], dh, c0, n0, m0, dc_last, c_states, cast_to,
                                           qk_scale, chunk_size, eps, impl, c0 is not None, reverse, siging, soft_cap,
                                           grad_dtype, normalize)
    # dN / dM_initial are zeros, as in native/bw.py:329-337 (and _MlstmChunkwiseB200)
    return (dq, dk, dv, di, df,
            None if c0 is None else dc0.to(cast_to if _autocast_eligible(c0) and cast_to else c0.dtype),
            None if n0 is None else torch.zeros_like(n0),
            None if m0 is None else torch.zeros_like(m0),
            None, None, None, None, None, None, None, None, None, None, None, None)


torch.library.register_autograd(chunkwise_fw, _chunkwise_backward, setup_context=_chunkwise_setup)


class _ChunkwiseFunction:
    """What ``backend._FUNCTIONS[kernel_dtype]`` is to eager calls: ``apply`` with ``_MlstmChunkwiseB200.forward``'s
    arguments (``siging`` the C-ABI mode 0 / 1 / 2), here over ``chunkwise_fw``."""

    def __init__(self, kernel_dtype):
        self.kernel_dtype = kernel_dtype

    def apply(self, q, k, v, i, f, c_initial, n_initial, m_initial, return_last_states, chunk_size, eps, reverse, siging,
              grad_dtype=None):
        cast_to = self.kernel_dtype if torch.is_autocast_enabled("cuda") else None
        dt = cast_to if (cast_to is not None and _autocast_eligible(q)) else q.dtype
        need_bw = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (q, k, v, i, f, c_initial))
        siging, normalize = _backend._siging_flags(siging)
        h, _, c_last, n_last, m_last, _ = chunkwise_fw(q, k, v, i, f, c_initial, n_initial, m_initial, cast_to, None,
                                                       return_last_states, chunk_size, eps, _backend._default_impl, need_bw,
                                                       reverse, siging, 0.0, grad_dtype, normalize)
        if not return_last_states:
            return h, None, None, None
        return h, c_last.to(dt), n_last.to(dt), m_last.to(dt)  # native kernels hand states back in the input dtype


_CHUNKWISE_FUNCTIONS = {dt: _ChunkwiseFunction(dt) for dt in _backend._FUNCTIONS}


def chunkwise_function(kernel_dtype) -> _ChunkwiseFunction:
    return _CHUNKWISE_FUNCTIONS[kernel_dtype]


def fw_launch(q, k, v, i, f, c0, n0, m0, qk_scale, return_last_states, chunk_size, eps, impl, save_states, reverse, siging,
              soft_cap=0.0):
    """``backend._fw_launch`` (without the fused epilogue) over ``chunkwise_fw``: what ``mlstm_chunkwise_fw`` calls
    (``siging`` the C-ABI mode 0 / 1 / 2)."""
    impl = _backend._default_impl if impl is None else impl
    q, k, v, i, f, c0, n0, m0 = (None if t is None else t.detach() for t in (q, k, v, i, f, c0, n0, m0))
    siging, normalize = _backend._siging_flags(siging)
    h, nm, c_last, n_last, m_last, c_states = chunkwise_fw(q, k, v, i, f, c0, n0, m0, None, qk_scale, return_last_states,
                                                           chunk_size, eps, impl, save_states, reverse, siging, soft_cap,
                                                           None, normalize)
    return h, nm, ((c_last, n_last, m_last) if return_last_states else None), (c_states if save_states else None)


def bw_launch(q, k, v, i, f, n_out, m_out, dh, c0, n0, m0, dc_last, qk_scale, chunk_size, eps, impl, want_dc_initial,
              c_states, reverse, siging, out, soft_cap, grad_dtype):
    """``mlstm_chunkwise_bw`` over ``chunkwise_bw`` (``siging`` the C-ABI mode 0 / 1 / 2).  Caller-provided ``out``
    tensors receive a copy of the gradients."""
    impl = _backend._default_impl if impl is None else impl
    if out is not None:
        grad_dtype = out[0].dtype
    args = (q, k, v, i, f, n_out, m_out, dh, c0, n0, m0, dc_last, c_states)
    args = tuple(None if t is None else t.detach() for t in args)
    siging, normalize = _backend._siging_flags(siging)
    dq, dk, dv, di, df, dc0 = chunkwise_bw(*args, None, qk_scale, chunk_size, eps, impl, want_dc_initial, reverse, siging,
                                           soft_cap, grad_dtype, normalize)
    if out is not None:
        for o, g in zip(out, (dq, dk, dv, di, df)):
            o.copy_(g)
        dq, dk, dv, di, df = out
    return dq, dk, dv, di, df, (dc0 if want_dc_initial else None)


# ------------------------------------------------------------------------------------------------------------------
# chunkwise mLSTM on the layer's own tensors: vil._MlstmLayerLayout and vil._MlstmCellFused
# ------------------------------------------------------------------------------------------------------------------
@_op("layer_fw")
def layer_fw(qk: Tensor, v: Tensor, gates: Tensor, NH: int, kernel_dtype: torch.dtype, chunk_size: int, eps: float,
             impl: int, save_states: bool, reverse: bool, siging: bool, soft_cap: float, grad_dtype: torch.dtype
             ) -> tuple[Tensor, Tensor, Tensor]:
    """The forward of ``vil._MlstmLayerLayout`` on qk (B, S, 2 NH DHQK) = [q | k], v (B, S, NH DHHV) and gates
    (B, S, 2 NH) = [i | f] (S a multiple of ``chunk_size``), rounded to ``kernel_dtype`` here.  Returns h
    (B, NH, S, DHHV), nm, c_states.  ``grad_dtype`` is read by the backward only."""
    _, h, nm, c_states = _vil._layer_fw(qk, v, gates, NH, kernel_dtype, chunk_size, eps, impl, save_states, reverse, siging,
                                        soft_cap)
    return h, nm, (c_states if c_states is not None else _empty(v, _U8))


@layer_fw.register_fake
def _(qk, v, gates, NH, kernel_dtype, chunk_size, eps, impl, save_states, reverse, siging, soft_cap, grad_dtype):
    B, S, _ = v.shape
    DK, DV = _vil._head_dims(qk, v, NH)
    nbytes = _states_bytes(B, NH, S, DK, DV, kernel_dtype, chunk_size, impl) if save_states else 0
    return (v.new_empty((B, NH, S, DV), dtype=kernel_dtype), v.new_empty((2, B, NH, S), dtype=_F32),
            v.new_empty(nbytes, dtype=_U8))


@_op("layer_bw")
def layer_bw(qk: Tensor, v: Tensor, gates: Tensor, nm: Tensor, dh: Tensor, c_states: Tensor, NH: int,
             kernel_dtype: torch.dtype, chunk_size: int, eps: float, impl: int, reverse: bool, siging: bool, soft_cap: float,
             grad_dtype: torch.dtype) -> tuple[Tensor, Tensor, Tensor]:
    """Gradients of ``layer_fw`` in the layer's layouts, written by the kernel in ``grad_dtype``: d_qk, d_v, d_gates."""
    return _vil._layer_bw(*_vil._kernel_tensors(qk, v, gates, kernel_dtype), nm.contiguous(), dh, _none(c_states), NH,
                          chunk_size, eps, impl, reverse, siging, soft_cap, grad_dtype)


@layer_bw.register_fake
def _(qk, v, gates, nm, dh, c_states, NH, kernel_dtype, chunk_size, eps, impl, reverse, siging, soft_cap, grad_dtype):
    return tuple(torch.empty_like(t, dtype=grad_dtype) for t in (qk, v, gates))


def _layer_setup(ctx, inputs, output):
    qk, v, gates, NH, kdt, chunk_size, eps, impl, _, reverse, siging, soft_cap, gdt = inputs
    ctx.save_for_backward(qk, v, gates, output[1], output[2])
    ctx.cfg = (NH, kdt, chunk_size, eps, impl, reverse, siging, soft_cap, gdt)
    ctx.set_materialize_grads(False)


def _layer_backward(ctx, dh, dnm, dc_states):
    qk, v, gates, nm, c_states = ctx.saved_tensors
    grads = layer_bw(qk, v, gates, nm, dh, c_states, *ctx.cfg)
    return (*_vil._to_dtypes(grads, (qk.dtype, v.dtype, gates.dtype)), None, None, None, None, None, None, None, None, None,
            None)


torch.library.register_autograd(layer_fw, _layer_backward, setup_context=_layer_setup)


@_op("chunkwise_fw_epilogue")
def chunkwise_fw_epilogue(qk: Tensor, v: Tensor, gates: Tensor, x_skip: Optional[Tensor], weight: Optional[Tensor],
                          bias: Optional[Tensor], skip: Optional[Tensor], NH: int, kernel_dtype: torch.dtype,
                          chunk_size: int, eps: float, impl: int, save_states: bool, reverse: bool, siging: bool,
                          soft_cap: float, ln_eps: float, out_dtype: torch.dtype, grad_dtype: torch.dtype
                          ) -> tuple[Tensor, Tensor, Tensor, Tensor]:
    """The forward of ``vil._MlstmCellFused``: ``layer_fw`` with MultiHeadLayerNorm, the relayout and the skip
    (``x_skip`` (B, S, H), or None) in the kernel's epilogue.  Returns y (B, S, NH DHHV), h (0-element unless
    ``save_states``: the LayerNorm backward reads it), nm, c_states."""
    _, _, y, h, nm, c_states = _vil._cell_fused_fw(qk, v, gates, x_skip, weight, bias, skip, NH, kernel_dtype, chunk_size,
                                                   eps, impl, save_states, reverse, siging, soft_cap, ln_eps, out_dtype)
    return (y, (h if h is not None else _empty(v, kernel_dtype)), nm,
            (c_states if c_states is not None else _empty(v, _U8)))


@chunkwise_fw_epilogue.register_fake
def _(qk, v, gates, x_skip, weight, bias, skip, NH, kernel_dtype, chunk_size, eps, impl, save_states, reverse, siging,
      soft_cap, ln_eps, out_dtype, grad_dtype):
    B, S, H = v.shape
    DK, DV = _vil._head_dims(qk, v, NH)
    h = v.new_empty((B, NH, S, DV) if save_states else (0,), dtype=kernel_dtype)
    nbytes = _states_bytes(B, NH, S, DK, DV, kernel_dtype, chunk_size, impl) if save_states else 0
    return v.new_empty((B, S, H), dtype=out_dtype), h, v.new_empty((2, B, NH, S), dtype=_F32), v.new_empty(nbytes, dtype=_U8)


def _epilogue_setup(ctx, inputs, output):
    qk, v, gates, xs, weight, bias, skip, NH, kdt, chunk_size, eps, impl, _, reverse, siging, soft_cap, ln_eps, out_dtype, \
        gdt = inputs
    ctx.save_for_backward(qk, v, gates, xs, weight, bias, skip, output[1], output[2], output[3])
    ctx.cfg = (NH, kdt, chunk_size, eps, impl, reverse, siging, soft_cap, gdt)
    ctx.ln = (ln_eps, out_dtype)
    ctx.set_materialize_grads(False)


def _epilogue_backward(ctx, dy, dh_unused, dnm, dc_states):
    qk, v, gates, xs, weight, bias, skip, h, nm, c_states = ctx.saved_tensors
    dh, dpar, dx = cellout_bw(h, xs, weight, skip, dy, *ctx.ln, ctx.needs_input_grad[3])
    grads = layer_bw(qk, v, gates, nm, dh, c_states, *ctx.cfg)
    return (*_vil._to_dtypes(grads, (qk.dtype, v.dtype, gates.dtype)), _none(dx),
            *_vil._param_grads(dpar, weight, bias, skip), None, None, None, None, None, None, None, None, None, None, None,
            None)


torch.library.register_autograd(chunkwise_fw_epilogue, _epilogue_backward, setup_context=_epilogue_setup)


# ------------------------------------------------------------------------------------------------------------------
# cell output, RMSNorm, convert16, recurrent sequence
# ------------------------------------------------------------------------------------------------------------------
@_op("cellout_fw")
def cellout_fw(h: Tensor, weight: Optional[Tensor], bias: Optional[Tensor], skip: Optional[Tensor], x: Optional[Tensor],
               eps: float, out_dtype: torch.dtype) -> Tensor:
    """``vil._CellOut``'s forward: y (B, S, NH D) in ``out_dtype``."""
    return _vil._cellout_fw_call(h, x, weight, bias, skip, eps, out_dtype)[0]


@cellout_fw.register_fake
def _(h, weight, bias, skip, x, eps, out_dtype):
    B, NH, S, D = h.shape
    return h.new_empty((B, S, NH * D), dtype=out_dtype)


@_op("cellout_bw")
def cellout_bw(h: Tensor, x: Optional[Tensor], weight: Optional[Tensor], skip: Optional[Tensor], dy: Tensor, eps: float,
               out_dtype: torch.dtype, want_dx: bool) -> tuple[Tensor, Tensor, Tensor]:
    """Returns dh (h's strides), dpar (3, H) fp32 = [dweight, dbias, dskip] and dx (0-element unless x and
    ``want_dx``)."""
    dh, dpar, dx = _vil._cellout_bw_call(h, x, weight, skip, dy, eps, out_dtype, want_dx)
    return dh, dpar, (dx if dx is not None else _empty(dy, out_dtype))


@cellout_bw.register_fake
def _(h, x, weight, skip, dy, eps, out_dtype, want_dx):
    B, NH, S, D = h.shape
    dx = dy.new_empty((B, S, NH * D), dtype=out_dtype) if (x is not None and want_dx) else _empty(dy, out_dtype)
    return (torch.empty_strided(h.shape, h.stride(), dtype=h.dtype, device=h.device),
            h.new_empty((3, NH * D), dtype=_F32), dx)


def _cellout_setup(ctx, inputs, output):
    h, weight, bias, skip, x, eps, out_dtype = inputs
    ctx.save_for_backward(h, x, weight, bias, skip)
    ctx.cfg = (eps, out_dtype)


def _cellout_backward(ctx, dy):
    h, x, weight, bias, skip = ctx.saved_tensors
    dh, dpar, dx = cellout_bw(h, x, weight, skip, dy, *ctx.cfg, ctx.needs_input_grad[4])
    return (dh, *_vil._param_grads(dpar, weight, bias, skip), _none(dx), None, None)


torch.library.register_autograd(cellout_fw, _cellout_backward, setup_context=_cellout_setup)


@_op("rmsnorm_fw")
def rmsnorm_fw(x2: Tensor, weight: Optional[Tensor], eps: float, out_dtype: torch.dtype) -> tuple[Tensor, Tensor]:
    """``vil._RmsNorm``'s forward on contiguous (rows, C) ``x2``: y (rows, C) in ``out_dtype``, rstd (rows,) fp32."""
    return _vil._rmsnorm_fw_call(x2, weight, eps, out_dtype)


@rmsnorm_fw.register_fake
def _(x2, weight, eps, out_dtype):
    return x2.new_empty(x2.shape, dtype=out_dtype), x2.new_empty(x2.shape[:1], dtype=_F32)


@_op("rmsnorm_bw")
def rmsnorm_bw(x2: Tensor, weight: Optional[Tensor], rstd: Tensor, dy2: Tensor, eps: float, out_dtype: torch.dtype
               ) -> tuple[Tensor, Tensor]:
    """dx (rows, C) in x2's dtype and dweight (C,) fp32."""
    return _vil._rmsnorm_bw_call(x2, weight, rstd, dy2, eps, out_dtype)


@rmsnorm_bw.register_fake
def _(x2, weight, rstd, dy2, eps, out_dtype):
    return torch.empty_like(x2), x2.new_empty(x2.shape[1:], dtype=_F32)


def _rmsnorm_setup(ctx, inputs, output):
    x2, weight, eps, out_dtype = inputs
    ctx.save_for_backward(x2, weight, output[1])
    ctx.cfg = (eps, out_dtype)
    ctx.set_materialize_grads(False)


def _rmsnorm_backward(ctx, dy, drstd):
    x2, weight, rstd = ctx.saved_tensors
    dx, dw = rmsnorm_bw(x2, weight, rstd, dy, *ctx.cfg)
    return dx, (None if weight is None else dw.to(weight.dtype)), None, None


torch.library.register_autograd(rmsnorm_fw, _rmsnorm_backward, setup_context=_rmsnorm_setup)


def rms_norm(x, weight, eps, out_dtype):
    """``vil._RmsNorm.apply`` over ``rmsnorm_fw`` / ``rmsnorm_bw``: the op takes (rows, C) and returns rstd too."""
    if not x.is_cuda:
        raise RuntimeError("rms_norm_b200: x is on the CPU; this backend has no CPU path")
    shp = x.shape
    y, _ = rmsnorm_fw(x.reshape(-1, shp[-1]).contiguous(), weight, float(eps), out_dtype)
    return y.view(shp)


@_op("convert16")
def _convert16(x: Tensor, dtype: torch.dtype) -> Tensor:
    """``backend.convert16`` between the two 16-bit dtypes (x.dtype != dtype)."""
    return _backend.convert16(x, dtype)


@_convert16.register_fake
def _(x, dtype):
    return torch.empty_like(x, dtype=dtype)  # the strides x.to(dtype) gives, and the kernel's (a dense x keeps them)


torch.library.register_autograd(_convert16, lambda ctx, dy: (convert16(dy, ctx.dtype), None),
                                setup_context=lambda ctx, inputs, output: setattr(ctx, "dtype", inputs[0].dtype))


def convert16(x, dtype):
    """``backend.convert16`` over the ``convert16`` op (16-bit CUDA tensors), ``x.to(dtype)`` otherwise."""
    if x.dtype is dtype:
        return x
    if not x.is_cuda or {x.dtype, dtype} != {torch.float16, torch.bfloat16} or x.numel() == 0:
        return x.to(dtype)
    return _convert16(x, dtype)


@_op("recurrent_sequence")
def _recurrent_sequence(q: Tensor, k: Tensor, v: Tensor, i: Tensor, f: Tensor, c_initial: Optional[Tensor],
                        n_initial: Optional[Tensor], m_initial: Optional[Tensor], return_last_states: bool, eps: float,
                        siging: bool, normalize: bool = True) -> tuple[Tensor, Tensor, Tensor, Tensor]:
    """``mlstm_recurrent_sequence__b200``: h and the last states fp32 (0-element unless ``return_last_states``)."""
    out = _backend.mlstm_recurrent_sequence__b200(q, k, v, i, f, c_initial, n_initial, m_initial, return_last_states, eps,
                                                  _F32, siging, normalize)
    if not return_last_states:
        return out, _empty(q), _empty(q), _empty(q)
    h, (c, n, m) = out
    return h, c, n, m


@_recurrent_sequence.register_fake
def _(q, k, v, i, f, c_initial, n_initial, m_initial, return_last_states, eps, siging, normalize=True):
    _backend._siging_mode(siging, normalize)
    B, NH, S, DK = q.shape
    DV = v.shape[-1]
    h = q.new_empty((B, NH, S, DV))
    if not return_last_states:
        return h, _empty(q), _empty(q), _empty(q)
    return (h, q.new_empty((B, NH, DK, DV), dtype=_F32), q.new_empty((B, NH, DK), dtype=_F32),
            q.new_empty((B, NH, 1), dtype=_F32))


def recurrent_sequence(q, k, v, i, f, c_initial, n_initial, m_initial, return_last_states, eps, dtype_state, siging,
                       normalize=True):
    """``mlstm_recurrent_sequence__b200`` over the ``recurrent_sequence`` op (forward only, like the eager call)."""
    args = tuple(None if t is None else t.detach() for t in (q, k, v, i, f, c_initial, n_initial, m_initial))
    h, c, n, m = _recurrent_sequence(*args, return_last_states, eps, siging, normalize)
    if not return_last_states:
        return h
    return h, (c.to(dtype_state), n.to(dtype_state), m.to(dtype_state))
