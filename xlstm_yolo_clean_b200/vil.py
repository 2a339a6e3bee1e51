"""Callers either side of the hot path (SURVEY.md section 8(f) #2, #3): the mLSTM branch of a ViLLayer with

  * the cell's output stage fused -- MultiHeadLayerNorm + (B,NH,S,D)->(B,S,H) relayout + learnable skip in one
    CUDA pass each way (C-ABI ``mlstm_b200_cellout_fw`` / ``_bw``) instead of group_norm + transposes + copies
    (ultralytics/nn/modules/vision_lstm/vision_lstm2.py:749-751, 928-944, 306);
  * the bottom-right scan direction without the two ``x.flip`` copies (vision_lstm2.py:292-294, 309-310): the
    kernel's anti-causal scan (``reverse=True``) plus the depthwise 3x3 conv evaluated with its weights rotated
    by 180 degrees, which is the same function because a flip of the row-major token sequence is a 180-degree
    rotation of the image and every other op on the branch acts per token;
  * the q/k/v/i/f views handed to the kernel as they are (BSHD-strided, no ``contiguous``), gradients written by
    the kernel straight into tensors of the layer's own layouts, no zero-padding copies for S = 400 / 100;
  * the two ``nn.RMSNorm`` modules in front of the branches (``ViLLayer.norm`` / ``.ffn_norm``, vision_lstm2.py:277-278,
    318-327) as one CUDA pass each way (``mlstm_b200_rmsnorm_fw`` / ``_bw``): under fp16 autocast torch's own falls off
    its fused path onto a composite of ~15 kernels per call.

``patch_model(model, fused=True)`` (backend.py) / ``patch_layers(model)`` rebind ``ViLLayer.mlstm_branch`` of the
reference model to ``mlstm_branch_b200`` and the two norms' ``forward`` to ``rms_norm_b200``; parameters, state-dict
keys and the function computed are unchanged.
PyTorch is used for the dense layers (cuBLAS / cuDNN serve them), device memory and autograd plumbing.
There is no CPU path: CPU tensors raise.
"""
from __future__ import annotations

import ctypes as C
import math

import torch
import torch.nn.functional as F

from . import _cabi
from . import backend as _backend
from . import ops as _ops
from torch.amp import custom_bwd, custom_fwd

from .backend import (_DTYPES, _cell_uses_siging, _on_device, _tensor, mlstm_chunkwise__b200, mlstm_siging_chunkwise__b200,
                      tensor_path_supported)


def cellout_supported(NH: int, D: int) -> bool:
    return D in (32, 64, 128) and (NH * D) % 128 == 0 and NH * D <= 2048


# one_launch="auto" for rectangular heads, by (DHQK, DHHV, gradients wanted): True = the cell as one forward launch (the
# rectangular forward with the fused epilogue, two-CTA clusters), False = the rectangular forward + cell-output pass.
# Measured on an NVIDIA B200 at 1000 W (profiles/r04_rect_epilogue_bench.jsonl, tools/rect_cell_bench.py; DESIGN.md
# section 4.3): the one-launch cell is 0-14 % slower without gradients and 17-38 % slower in training at both pairs and
# both BASELINE call sizes, so "auto" keeps two launches; one_launch="always" still fuses.
RECT_ONE_LAUNCH = {
    (32, 64, False): False, (32, 64, True): False,
    (64, 128, False): False, (64, 128, True): False,
}


def _f32c(t):
    return None if t is None else t.detach().to(torch.float32).contiguous()


def _vec_ok(t: torch.Tensor) -> bool:
    return t.stride(-1) == 1 and all(s % 4 == 0 for s in t.stride()[:-1]) and t.data_ptr() % 16 == 0


def _rows(t, dtype):
    """x, y, dy and dx of the cell-output kernels and of the fused epilogue move as dense (B, S, H) rows in the output
    dtype at a 16-byte-aligned address: ``t`` as such rows, copied where it is not (None stays None)."""
    if t is None or (t.dtype == dtype and t.is_contiguous() and t.data_ptr() % 16 == 0):
        return t
    t = t.to(dtype).contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()  # a contiguous view at an odd offset of its storage


def _param_grads(dpar, weight, bias, skip):
    """Gradients of weight / bias / skip from dpar (3, H) fp32 = [dweight, dbias, dskip], in the parameters' dtypes."""
    return tuple(None if p is None else g.to(p.dtype) for g, p in zip(dpar, (weight, bias, skip)))


def _to_dtypes(grads, dtypes):
    return tuple(g if g.dtype == dt else g.to(dt) for g, dt in zip(grads, dtypes))


def _cellout_fw_call(h, x, weight, bias, skip, eps, out_dtype):
    """mlstm_b200_cellout_fw: y (B, S, NH*D) in ``out_dtype``, and the h and x the kernel read (h copied where it fails
    ``_vec_ok``, x as ``_rows``)."""
    lib = _cabi.load_library()
    h = h if _vec_ok(h) else h.contiguous()
    x = _rows(x, out_dtype)
    B, NH, S, D = h.shape
    w32, b32, s32 = _f32c(weight), _f32c(bias), _f32c(skip)
    with _on_device(h.device):
        y = torch.empty(B, S, NH * D, dtype=out_dtype, device=h.device)
        a = _cabi.CellOutArgs()
        a.B, a.NH, a.S, a.D = B, NH, S, D
        a.h_dtype, a.x_dtype, a.y_dtype = _DTYPES[h.dtype], _DTYPES[out_dtype], _DTYPES[out_dtype]
        a.eps = float(eps)
        a.h, a.x, a.y = _tensor(h), _tensor(x), _tensor(y)
        a.weight = None if w32 is None else w32.data_ptr()
        a.bias = None if b32 is None else b32.data_ptr()
        a.skip = None if s32 is None else s32.data_ptr()
        st = lib.mlstm_b200_cellout_fw(C.byref(a), C.c_void_p(torch.cuda.current_stream(h.device).cuda_stream))
        _cabi.check(st, "mlstm_b200_cellout_fw")
    return y, h, x


def _cellout_bw_call(h, x, weight, skip, dy, eps, out_dtype, want_dx):
    """mlstm_b200_cellout_bw: returns dh (h's strides), dpar (3, H) fp32 = [dweight, dbias, dskip] and dx (None unless x
    and ``want_dx``).  h and x are prepared as in the forward, so the saved inputs of either one can be passed."""
    lib = _cabi.load_library()
    hk = h if _vec_ok(h) else h.contiguous()
    x, dy = _rows(x, out_dtype), _rows(dy, out_dtype)
    B, NH, S, D = h.shape
    w32, s32 = _f32c(weight), _f32c(skip)
    dev = h.device
    with _on_device(dev):
        dh = torch.empty_strided(hk.shape, hk.stride(), dtype=h.dtype, device=dev)  # the kernel walks h and dh together
        dx = torch.empty_like(dy) if (x is not None and want_dx) else None
        dpar = torch.empty(3, NH * D, dtype=torch.float32, device=dev)
        b = _cabi.CellOutBwArgs()
        a = b.fw
        a.B, a.NH, a.S, a.D = B, NH, S, D
        a.h_dtype, a.x_dtype, a.y_dtype = _DTYPES[h.dtype], _DTYPES[out_dtype], _DTYPES[out_dtype]
        a.eps = eps
        a.h, a.x = _tensor(hk), _tensor(x)
        a.weight = None if w32 is None else w32.data_ptr()
        a.skip = None if s32 is None else s32.data_ptr()
        b.dy, b.dh, b.dx = _tensor(dy), _tensor(dh), _tensor(dx)
        b.dweight, b.dbias, b.dskip = dpar[0].data_ptr(), dpar[1].data_ptr(), dpar[2].data_ptr()
        ws_bytes = lib.mlstm_b200_cellout_workspace_bytes(C.byref(a))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        b.workspace, b.workspace_bytes = ws.data_ptr(), ws_bytes
        st = lib.mlstm_b200_cellout_bw(C.byref(b), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
        _cabi.check(st, "mlstm_b200_cellout_bw")
    if hk is not h:
        dh = torch.empty_strided(h.shape, h.stride(), dtype=h.dtype, device=dev).copy_(dh)
    return dh, dpar, dx


class _CellOut(torch.autograd.Function):
    """y = MultiHeadLayerNorm(h) [+ skip * x], h (B,NH,S,D) -> y (B,S,NH*D)."""

    @staticmethod
    def forward(ctx, h, weight, bias, skip, x, eps, out_dtype):
        y, h, x = _cellout_fw_call(h, x, weight, bias, skip, eps, out_dtype)
        ctx.save_for_backward(h, x, weight, bias, skip)
        ctx.eps, ctx.out_dtype = float(eps), out_dtype
        return y

    @staticmethod
    def backward(ctx, dy):
        h, x, weight, bias, skip = ctx.saved_tensors
        dh, dpar, dx = _cellout_bw_call(h, x, weight, skip, dy, ctx.eps, ctx.out_dtype, ctx.needs_input_grad[4])
        return (dh, *_param_grads(dpar, weight, bias, skip), dx, None, None)


def cell_out(h, weight=None, bias=None, skip=None, x=None, eps=1e-6, out_dtype=None):
    """Fused MultiHeadLayerNorm (+ skip): see the module docstring.  ``weight`` is the effective scale
    (the reference's ``weight_proxy`` = 1 + weight, vision_lstm2.py:900-907)."""
    out_dtype = out_dtype or (x.dtype if x is not None else h.dtype)
    if not h.is_cuda:
        raise RuntimeError("cell_out: h is on the CPU; this backend has no CPU path")
    if torch.compiler.is_compiling():
        return _ops.cellout_fw(h, weight, bias, skip, x, float(eps), out_dtype)
    return _CellOut.apply(h, weight, bias, skip, x, eps, out_dtype)


RMSNORM_DIMS = (192, 256, 384, 512)


def _rmsnorm_fw_call(x2, weight, eps, out_dtype):
    """mlstm_b200_rmsnorm_fw on contiguous (rows, C) ``x2``: returns y (rows, C) in ``out_dtype`` and rstd (rows,) fp32."""
    lib = _cabi.load_library()
    rows, Cdim = x2.shape
    w32 = _f32c(weight)
    with _on_device(x2.device):
        y = torch.empty(rows, Cdim, dtype=out_dtype, device=x2.device)
        rstd = torch.empty(rows, dtype=torch.float32, device=x2.device)
        a = _cabi.RmsNormArgs()
        a.rows, a.C, a.x_dtype, a.y_dtype, a.eps = rows, Cdim, _DTYPES[x2.dtype], _DTYPES[out_dtype], float(eps)
        a.x, a.y, a.rstd = x2.data_ptr(), y.data_ptr(), rstd.data_ptr()
        a.weight = None if w32 is None else w32.data_ptr()
        st = lib.mlstm_b200_rmsnorm_fw(C.byref(a), C.c_void_p(torch.cuda.current_stream(x2.device).cuda_stream))
        _cabi.check(st, "mlstm_b200_rmsnorm_fw")
    return y, rstd


def _rmsnorm_bw_call(x2, weight, rstd, dy, eps, out_dtype):
    """mlstm_b200_rmsnorm_bw: dx (rows, C) in x2's dtype and dweight (C,) fp32; ``dy`` has x2's number of elements and
    is read as contiguous (rows, C) in ``out_dtype``."""
    lib = _cabi.load_library()
    rows, Cdim = x2.shape
    dy2 = dy.reshape(rows, Cdim)
    dy2 = dy2 if (dy2.dtype == out_dtype and dy2.is_contiguous()) else dy2.to(out_dtype).contiguous()
    w32 = _f32c(weight)
    dev = x2.device
    with _on_device(dev):
        dx = torch.empty_like(x2)
        dw = torch.empty(Cdim, dtype=torch.float32, device=dev)
        b = _cabi.RmsNormBwArgs()
        a = b.fw
        a.rows, a.C, a.x_dtype, a.y_dtype, a.eps = rows, Cdim, _DTYPES[x2.dtype], _DTYPES[out_dtype], eps
        a.x, a.rstd = x2.data_ptr(), rstd.data_ptr()
        a.weight = None if w32 is None else w32.data_ptr()
        b.dy, b.dx, b.dweight = dy2.data_ptr(), dx.data_ptr(), dw.data_ptr()
        nws = lib.mlstm_b200_rmsnorm_workspace_bytes(C.byref(a))
        ws = torch.empty(nws, dtype=torch.uint8, device=dev)
        b.workspace, b.workspace_bytes = ws.data_ptr(), nws
        st = lib.mlstm_b200_rmsnorm_bw(C.byref(b), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
        _cabi.check(st, "mlstm_b200_rmsnorm_bw")
    return dx, dw


class _RmsNorm(torch.autograd.Function):
    """nn.RMSNorm over the last dimension (ViLLayer.norm / .ffn_norm, vision_lstm2.py:277-278) as one CUDA pass each
    way.  ``out_dtype``: what the consumer reads (a Linear under autocast reads the autocast dtype)."""

    @staticmethod
    def forward(ctx, x, weight, eps, out_dtype):
        if not x.is_cuda:
            raise RuntimeError("rms_norm_b200: x is on the CPU; this backend has no CPU path")
        shp = x.shape
        x2 = x.reshape(-1, shp[-1])
        x2 = x2 if x2.is_contiguous() else x2.contiguous()
        y, rstd = _rmsnorm_fw_call(x2, weight, eps, out_dtype)
        ctx.save_for_backward(x2, weight, rstd)
        ctx.eps, ctx.out_dtype, ctx.shp = float(eps), out_dtype, shp
        return y.view(shp)

    @staticmethod
    def backward(ctx, dy):
        x2, weight, rstd = ctx.saved_tensors
        dx, dw = _rmsnorm_bw_call(x2, weight, rstd, dy, ctx.eps, ctx.out_dtype)
        return dx.view(ctx.shp), (None if weight is None else dw.to(weight.dtype)), None, None


def rms_norm_b200(x, weight=None, eps=1e-6, out_dtype=None):
    """Fused RMSNorm.  Default ``out_dtype``: the CUDA autocast dtype if autocast is on (the consumers in ViLLayer
    are Linear layers, which read exactly that), else the input dtype like torch.rms_norm."""
    if out_dtype is None:
        if torch.is_autocast_enabled("cuda"):
            out_dtype = torch.get_autocast_dtype("cuda")
        else:
            out_dtype = x.dtype  # torch.rms_norm returns the input dtype
    if torch.compiler.is_compiling():
        return _ops.rms_norm(x, weight, eps, out_dtype)
    return _RmsNorm.apply(x, weight, eps, out_dtype)


TENSOR_HEAD_DIMS = ((32, 32), (64, 64), (128, 128), (32, 64), (64, 128))  # (DHQK, DHHV) of the tensor-core kernels


def _head_dims(qk, v, NH):
    """(DHQK, DHHV) of layer-layout tensors: qk (B, S, 2 NH DHQK) = [q | k], v (B, S, NH DHHV)."""
    return qk.shape[-1] // (2 * NH), v.shape[-1] // NH


def _layer_grad_dtype(in_dtypes, kernel_dtype, head_dims, S):
    """``backend._grad_dtype`` of a layer-layout call: the dtype the layer's tensors had before they were re-rounded to
    the kernel dtype (fp16 under ultralytics' AMP with the bf16 kernels) when the three agree, on the tensor-core route
    as the head dims, S and the implementation choice determine it (no query)."""
    dt = in_dtypes[0]
    caller = dt if all(t is dt for t in in_dtypes) else None
    tensor_route = head_dims in TENSOR_HEAD_DIMS and S % 4 == 0 and _backend._default_impl != _cabi.IMPL_EXACT
    return _backend._grad_dtype(kernel_dtype, caller, tensor_route)


@torch.compiler.assume_constant_result
def _tensor_path_supported(NH: int, S: int, DK: int, DV: int, dtype: torch.dtype, chunk_size: int) -> bool:
    """``backend.tensor_path_supported`` for B = 1 (the support matrix does not depend on B), a constant while
    torch.compile traces."""
    return tensor_path_supported(1, NH, S, DK, DV, dtype, chunk_size)


def _layer_chunking(S, NH, head_dims, chunk_size, kernel_dtype):
    """(chunk_size, pad) of a layer-layout call.  The tcgen05 kernels walk 128-token tiles whatever the chunk size is
    and handle a ragged last tile themselves (the result does not depend on chunk_size: the stabiliser equals the
    step-recurrent one), so on the tensor-core route S = 400 / 100 run as they are with a chunk size that divides them;
    elsewhere the tensors are zero-padded to a multiple of ``chunk_size``."""
    if S % chunk_size and kernel_dtype in (torch.float16, torch.bfloat16):
        g = math.gcd(S, chunk_size)
        if _tensor_path_supported(NH, S, *head_dims, kernel_dtype, g):
            chunk_size = g
    return chunk_size, (-S) % chunk_size


def _heads(qk, v, gates, NH):
    """(B, NH, S, DHQK) q / k, (B, NH, S, DHHV) v and (B, NH, S) i / f views of the layer-layout tensors: no data
    movement.  q / k may be narrower than v (rectangular heads)."""
    B, S, H = v.shape
    DK, DV = _head_dims(qk, v, NH)
    Hqk = NH * DK
    q = qk[..., :Hqk].view(B, S, NH, DK).transpose(1, 2)
    k = qk[..., Hqk:].view(B, S, NH, DK).transpose(1, 2)
    vv = v.view(B, S, NH, DV).transpose(1, 2)
    return q, k, vv, gates[..., :NH].transpose(1, 2), gates[..., NH:].transpose(1, 2)


def _kernel_tensors(qk, v, gates, kernel_dtype):
    return tuple(_backend.convert16(t, kernel_dtype) for t in (qk, v, gates))  # (fp32 inputs: torch's cast)


def _layer_fw(qk, v, gates, NH, kernel_dtype, chunk_size, eps, impl, save_states, reverse, siging, soft_cap, epi=None):
    """Forward of the chunkwise mLSTM on the layer's tensors (S a multiple of ``chunk_size``), rounded to
    ``kernel_dtype`` here; ``epi``: the fused cell-output epilogue.  Returns the rounded (qk, v, gates), h, nm, c_states."""
    ts = _kernel_tensors(qk, v, gates, kernel_dtype)
    h, nm, _, c_states = _backend._fw_launch(*_heads(*ts, NH), None, None, None, None, False, chunk_size, eps, impl,
                                             save_states, reverse, siging, soft_cap, epi)
    return ts, h, nm, c_states


def _layer_bw(qk, v, gates, nm, dh, c_states, NH, chunk_size, eps, impl, reverse, siging, soft_cap, grad_dtype):
    """Gradients of ``_layer_fw`` from its rounded tensors, written by the kernel in ``grad_dtype`` straight into
    tensors of the layer's layouts: d_qk, d_v, d_gates."""
    grads = tuple(torch.empty_like(t, dtype=grad_dtype) for t in (qk, v, gates))
    n_ptr, m_ptr = _backend._nm_ptrs(nm)
    _backend._bw_launch(*_heads(qk, v, gates, NH), n_ptr, m_ptr, dh, None, None, None, None, None, chunk_size, eps, impl,
                        False, c_states, reverse, siging, _heads(*grads, NH), soft_cap)
    return grads


class _MlstmLayerLayout(torch.autograd.Function):
    """Chunkwise mLSTM on the tensors the layer already owns -- qk (B, S, 2H) = [q | k] from qk_proj, v (B, S, H),
    gates (B, S, 2NH) = [i | f] -- with the gradients written by the kernel straight into tensors of those
    layouts.  Same C-ABI calls as ``mlstm_chunkwise__b200``; what disappears is the autograd glue around
    (B, NH, S, D) tensors: three transpose-copies and the q/k concatenation in every backward."""

    @staticmethod
    @custom_fwd(device_type="cuda")
    def forward(ctx, qk, v, gates, NH, kernel_dtype, chunk_size, eps, impl, reverse, siging, soft_cap, grad_dtype):
        ts, h, nm, c_states = _layer_fw(qk, v, gates, NH, kernel_dtype, chunk_size, eps, impl,
                                        any(ctx.needs_input_grad[:3]), reverse, siging, soft_cap)
        ctx.save_for_backward(*ts, nm, c_states)
        ctx.cfg = (NH, chunk_size, eps, impl, reverse, siging, soft_cap, grad_dtype)
        ctx.in_dtypes = (qk.dtype, v.dtype, gates.dtype)
        return h

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, dh):
        qk_k, v_k, g_k, nm, c_states = ctx.saved_tensors
        grads = _layer_bw(qk_k, v_k, g_k, nm, dh, c_states, *ctx.cfg)
        return (*_to_dtypes(grads, ctx.in_dtypes), None, None, None, None, None, None, None, None, None)


def _layer_layout(qk, v, gates, NH, reverse, siging, chunk_size, eps, kernel_dtype, soft_cap):
    """h (B, NH, S, DHHV) of the chunkwise mLSTM on the layer's tensors: ``_MlstmLayerLayout``, or the ``layer_fw`` op
    while torch.compile traces."""
    S = v.shape[1]
    head_dims = _head_dims(qk, v, NH)
    chunk_size, pad = _layer_chunking(S, NH, head_dims, chunk_size, kernel_dtype)
    gdt = _layer_grad_dtype((qk.dtype, v.dtype, gates.dtype), kernel_dtype, head_dims, S + pad)
    if pad:  # zero padding as wrap_chunkwise__pad_zeros (kernel_wrappers.py:227-247); padded tokens come last
        pp = (0, 0, pad, 0) if reverse else (0, 0, 0, pad)  # in scan order = first in memory when reversed
        qk, v, gates = (F.pad(t, pp) for t in (qk, v, gates))
    args = (qk, v, gates, NH, kernel_dtype, chunk_size, eps, _backend._default_impl)
    if torch.compiler.is_compiling():
        need_bw = torch.is_grad_enabled() and any(t.requires_grad for t in (qk, v, gates))
        h = _ops.layer_fw(*args, need_bw, reverse, siging, soft_cap, gdt)[0]
    else:
        h = _MlstmLayerLayout.apply(*args, reverse, siging, soft_cap, gdt)
    if pad:
        h = h[:, :, pad:] if reverse else h[:, :, :S]
    return h


def _cell_fused_fw(qk, v, gates, x_skip, weight, bias, skip, NH, kernel_dtype, chunk_size, eps, impl, save_states, reverse,
                   siging, soft_cap, ln_eps, out_dtype):
    """``_layer_fw`` with MultiHeadLayerNorm, the relayout and the skip (``x_skip`` prepared as ``_rows``, or None) in
    the kernel's epilogue.  Returns the rounded (qk, v, gates), the skip input read, y (B, S, NH DHHV), h (None unless
    ``save_states``: the LayerNorm backward reads it), nm, c_states."""
    B, S, H = v.shape
    D = H // NH
    xs = _rows(x_skip, out_dtype)
    y = torch.empty(B, S, H, dtype=out_dtype, device=v.device)
    as_heads = lambda t: t.view(B, S, NH, D).transpose(1, 2)  # noqa: E731  (B, NH, S, D) view of a (B, S, H) tensor
    epi = _backend.FwEpilogue(as_heads(y), None if xs is None else as_heads(xs), _f32c(weight), _f32c(bias),
                              None if xs is None else _f32c(skip), ln_eps, save_states)
    ts, h, nm, c_states = _layer_fw(qk, v, gates, NH, kernel_dtype, chunk_size, eps, impl, save_states, reverse, siging,
                                    soft_cap, epi)
    return ts, xs, y, h, nm, c_states


class _MlstmCellFused(torch.autograd.Function):
    """The whole cell in ONE forward launch (SURVEY.md section 8(f) #3): chunkwise mLSTM on the layer's own tensors (like
    ``_MlstmLayerLayout``) with MultiHeadLayerNorm, the (B, NH, S, D) -> (B, S, H) relayout and the learnable skip done in
    the kernel's epilogue (C-ABI ``mlstm_b200_fw_epilogue``): no separate cell-output pass, and under no_grad h never
    reaches HBM un-normalised.  In training h is also written (the LayerNorm backward needs it); the backward is the
    stand-alone cell-output backward (over DHHV) followed by the mLSTM backward.  q / k may be narrower than v."""

    @staticmethod
    @custom_fwd(device_type="cuda")
    def forward(ctx, qk, v, gates, x_skip, weight, bias, skip, NH, kernel_dtype, chunk_size, eps, impl, reverse, siging,
                soft_cap, ln_eps, out_dtype, grad_dtype):
        ts, xs, y, h, nm, c_states = _cell_fused_fw(qk, v, gates, x_skip, weight, bias, skip, NH, kernel_dtype, chunk_size,
                                                    eps, impl, any(ctx.needs_input_grad[:7]), reverse, siging, soft_cap,
                                                    ln_eps, out_dtype)
        ctx.save_for_backward(*ts, nm, c_states, h, xs, weight, bias, skip)
        ctx.cfg = (NH, chunk_size, eps, impl, reverse, siging, soft_cap, grad_dtype)
        ctx.ln = (ln_eps, out_dtype)
        ctx.in_dtypes = (qk.dtype, v.dtype, gates.dtype)
        return y

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, dy):
        qk_k, v_k, g_k, nm, c_states, h, xs, weight, bias, skip = ctx.saved_tensors
        dh, dpar, dx = _cellout_bw_call(h, xs, weight, skip, dy, *ctx.ln, ctx.needs_input_grad[3])
        grads = _layer_bw(qk_k, v_k, g_k, nm, dh, c_states, *ctx.cfg)
        return (*_to_dtypes(grads, ctx.in_dtypes), dx, *_param_grads(dpar, weight, bias, skip),
                None, None, None, None, None, None, None, None, None, None, None)


def _cell_fused(qk, v, gates, x_skip, weight, bias, skip, NH, reverse, siging, chunk_size, eps, kernel_dtype, soft_cap,
                ln_eps, out_dtype):
    """y (B, S, NH DHHV) of the one-launch cell: ``_MlstmCellFused``, or the ``chunkwise_fw_epilogue`` op while
    torch.compile traces.  The skip is added only with both ``skip`` and ``x_skip``."""
    S = v.shape[1]
    head_dims = _head_dims(qk, v, NH)
    chunk_size, pad = _layer_chunking(S, NH, head_dims, chunk_size, kernel_dtype)
    if pad:
        raise RuntimeError("the fused cell-output epilogue exists on the tensor-core route only")
    if x_skip is None or skip is None:
        x_skip = skip = None
    gdt = _layer_grad_dtype((qk.dtype, v.dtype, gates.dtype), kernel_dtype, head_dims, S)
    args = (qk, v, gates, x_skip, weight, bias, skip, NH, kernel_dtype, chunk_size, eps, _backend._default_impl)
    if torch.compiler.is_compiling():
        need_bw = torch.is_grad_enabled() and any(
            t is not None and t.requires_grad for t in (qk, v, gates, x_skip, weight, bias, skip))
        return _ops.chunkwise_fw_epilogue(*args, need_bw, reverse, siging, soft_cap, ln_eps, out_dtype, gdt)[0]
    return _MlstmCellFused.apply(*args, reverse, siging, soft_cap, ln_eps, out_dtype, gdt)


def _is_reverse(layer) -> bool:
    d = getattr(layer, "direction", None)
    name = getattr(d, "name", None) or getattr(d, "value", None) or str(d)
    return "BOT_RIGHT" in str(name).upper()


def _seq_conv(conv, x, rotate: bool):
    """SequenceConv2d (vision_lstm_util.py:96-114) on (B, S, C) tokens; ``rotate`` evaluates it with the
    kernel rotated by 180 degrees = conv(flip(x)) flipped back."""
    B, S, Cc = x.shape
    seqlens = getattr(conv, "seqlens", None)
    hh = int(seqlens[0]) if seqlens is not None else int(round(S ** 0.5))
    w = conv.weight.flip(-1, -2) if rotate else conv.weight
    img = x.view(B, hh, S // hh, Cc).permute(0, 3, 1, 2)
    out = F.conv2d(img, w, conv.bias, conv.stride, conv.padding, conv.dilation, conv.groups)
    return out.permute(0, 2, 3, 1).reshape(B, S, Cc)


def _gate_preact(cell, q, k, v, qk=None):
    """ifgate(cat[q, k, v]) (vision_lstm2.py:711-714).  When the caller still holds the fused qk_proj output
    ``qk`` (B, S, 2H) whose halves q and k are, the (B, S, 3H) concatenation is never materialised: the product
    splits into two GEMMs over tensors that already exist, accumulated inside the second one (addmm)."""
    if qk is None:
        return cell.ifgate(torch.cat([q, k, v], dim=-1))
    B, S, H2 = qk.shape
    W, b = cell.ifgate.weight, cell.ifgate.bias
    pre_v = F.linear(v, W[:, H2:], b)
    return torch.addmm(pre_v.reshape(B * S, -1), qk.reshape(B * S, H2), W[:, :H2].t()).view(B, S, -1)


def mlstm_cell_b200(cell, q, k, v, reverse=False, skip=None, x_skip=None, siging=False, chunk_size=64, eps=1e-6,
                    kernel_dtype="bfloat16", qk=None, one_launch="auto"):
    """MatrixLSTMCell.forward (vision_lstm2.py:701-753) on the B200 kernels, output stage fused.

    q, k, v (B, S, H) -> (B, S, H).  ``reverse`` runs the anti-causal scan; ``skip`` / ``x_skip`` add
    ViLLayer's ``learnable_skip * x_qk_conv_act`` inside the same pass.  Kernel parameters are the ones the
    reference's pad wrapper forces on every call: chunk 64, eps 1e-6, bf16 under CUDA autocast
    (kernel_wrappers.py:214-217; SURVEY.md finding 3).  ``kernel_dtype="input"`` is an opt-in deviation: 16-bit
    inputs go to the kernel as they are (fp16 under ultralytics' AMP) instead of being re-rounded to bf16, which
    drops five cast passes forward and five backward; the result is closer to the fp32 function, not identical
    to the reference's bf16 one.  ``one_launch``: "auto" | "always" | "never" -- when the cell runs as ONE forward launch
    (fused LayerNorm / skip epilogue); see below."""
    if one_launch not in ("auto", "always", "never"):
        raise ValueError(f"one_launch must be 'auto', 'always' or 'never' (got {one_launch!r})")
    B, S, H = v.shape  # q / k (B, S, NH DHQK) may be narrower than v (B, S, NH DHHV); the output is v's width
    if not q.is_cuda:
        raise RuntimeError("mlstm_cell_b200: tensors are on the CPU; this backend has no CPU path")
    NH = cell.num_heads
    DK, D = q.shape[-1] // NH, H // NH
    if_preact = _gate_preact(cell, q, k, v, qk)
    model_dtype = q.dtype
    if qk is not None:  # layer-layout path: the kernel reads / writes the layer's own tensors
        autocast_on = torch.is_autocast_enabled("cuda")
        in_dt = cell.autocast_dtype if cell.use_autocast else qk.dtype  # the reference casts on CUDA in train and eval
        kdt = in_dt if (not autocast_on or (kernel_dtype == "input" and in_dt in (torch.float16, torch.bfloat16))) \
            else torch.bfloat16  # custom_fwd(cast_inputs=bf16) rule of the registry kernels (native/fwbw.py:37)
        # soft_cap (vision_lstm2.py:714-715, 755-756): on the tensor-core route the scan warp of the kernels applies
        # cap * tanh(x / cap) to the pre-activations it reads anyway, and the backward applies its derivative where it
        # stores dI / dF -- no elementwise passes over the gates in either direction (zero padding stays zero: tanh 0 = 0)
        in_kernel_cap = (kdt in (torch.float16, torch.bfloat16) and (DK, D) in TENSOR_HEAD_DIMS
                         and _backend._default_impl != _cabi.IMPL_EXACT)
        gates = if_preact if in_kernel_cap else cell.gate_soft_cap * torch.tanh(if_preact / cell.gate_soft_cap)
        qk_c, v_c, g_c = qk, v, gates
        if cell.use_autocast:
            qk_c, v_c, g_c = (t.to(cell.autocast_dtype) for t in (qk_c, v_c, g_c))
        norm = cell.outnorm
        out_dtype = torch.get_autocast_dtype("cuda") if autocast_on else model_dtype
        # One launch for the whole cell (_MlstmCellFused: the kernel's epilogue normalises, relayouts and adds the skip)
        # where that is the faster composition -- measured on B200 (DESIGN.md section 4.3): without gradients at head
        # dims 32 / 64 (h never reaches HBM: 334 vs 397 us at 256 heads x 6400 x 64).  In training h has to be written
        # as well (the LayerNorm backward reads it) and at head dim 128 the epilogue holds 64 columns per thread; there
        # the mLSTM kernel followed by the stand-alone cell-output pass is faster (408 vs 428 us; 327 vs 352 us).
        needs_grad = torch.is_grad_enabled() and any(
            t is not None and t.requires_grad for t in (qk_c, v_c, g_c, x_skip, norm.weight_proxy, norm.bias, skip))
        if DK == D:
            auto_fuse = not needs_grad and D in (32, 64)
        else:  # rectangular heads: RECT_ONE_LAUNCH, measured separately (the epilogue runs as two-CTA clusters)
            auto_fuse = RECT_ONE_LAUNCH.get((DK, D, needs_grad), False)
        fuse = one_launch == "always" or (one_launch == "auto" and auto_fuse)
        if (fuse and in_kernel_cap and S % 4 == 0 and out_dtype in (torch.float16, torch.bfloat16)
                and cellout_supported(NH, D) and (x_skip is None or x_skip.shape == (B, S, H))):
            return _cell_fused(qk_c, v_c, g_c, x_skip, norm.weight_proxy, norm.bias, skip, NH, bool(reverse), bool(siging),
                               int(chunk_size), float(eps), kdt, float(cell.gate_soft_cap), float(norm.eps), out_dtype)
        h = _layer_layout(qk_c, v_c, g_c, NH, bool(reverse), bool(siging), int(chunk_size), float(eps), kdt,
                          float(cell.gate_soft_cap) if in_kernel_cap else 0.0)
    else:
        capped = cell.gate_soft_cap * torch.tanh(if_preact / cell.gate_soft_cap)  # soft_cap, vision_lstm2.py:755-756
        i_pre, f_pre = torch.chunk(capped, 2, dim=-1)
        i, f = i_pre.transpose(-1, -2), f_pre.transpose(-1, -2)  # (B, NH, S) views
        qh, kh, vh = (t.view(B, S, NH, t.shape[-1] // NH).transpose(1, 2) for t in (q, k, v))  # (B, NH, S, D) views, no copy
        if cell.use_autocast:
            qh, kh, vh, i, f = (t.to(cell.autocast_dtype) for t in (qh, kh, vh, i, f))
        pad = (-S) % chunk_size
        if pad:  # zero padding like wrap_chunkwise__pad_zeros (kernel_wrappers.py:227-247); the padded tokens must
            # come LAST in scan order, i.e. at the front of memory for the anti-causal direction
            pq = (0, 0, pad, 0) if reverse else (0, 0, 0, pad)
            pg = (pad, 0) if reverse else (0, pad)
            qh, kh, vh = (F.pad(t, pq) for t in (qh, kh, vh))
            i, f = F.pad(i, pg), F.pad(f, pg)
        fn = mlstm_siging_chunkwise__b200 if siging else mlstm_chunkwise__b200
        kdt = qh.dtype if (kernel_dtype == "input" and qh.dtype in (torch.float16, torch.bfloat16)) else torch.bfloat16
        h = fn(q=qh, k=kh, v=vh, i=i, f=f, chunk_size=chunk_size, eps=eps, autocast_kernel_dtype=kdt, reverse=reverse)
        if pad:
            h = h[:, :, pad:] if reverse else h[:, :, :S]
    norm = cell.outnorm
    out_dtype = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else model_dtype
    return cell_out(h, norm.weight_proxy, norm.bias, skip, x_skip, eps=norm.eps, out_dtype=out_dtype)


def mlstm_branch_b200(layer, x, siging=False, kernel_dtype="bfloat16", one_launch="auto"):
    """ViLLayer.mlstm_branch (vision_lstm2.py:292-312) without flips and with the fused cell output."""
    rev = _is_reverse(layer)
    x_inner = layer.proj_up(x)
    x_qk, x_v = torch.chunk(x_inner, 2, dim=-1)
    if isinstance(layer.conv, torch.nn.Conv2d):
        x_act = F.silu(_seq_conv(layer.conv, x_qk, rotate=rev))
    else:
        x_act = F.silu(layer.conv(x_qk))
    qk = layer.qk_proj(x_act)
    q, k = torch.chunk(qk, 2, dim=-1)
    v = layer.v_proj(x_v)
    y = mlstm_cell_b200(layer.mlstm_cell, q, k, v, reverse=rev, skip=layer.learnable_skip, x_skip=x_act, siging=siging,
                        kernel_dtype=kernel_dtype, qk=qk, one_launch=one_launch)
    return layer.proj_down(y)


def _branch_entry(layer, x, siging=False, kernel_dtype="bfloat16", one_launch="auto"):
    """What ``patch_layers`` binds as ``layer.mlstm_branch`` (module-level, so that a patched model pickles)."""
    return mlstm_branch_b200(layer, x, siging=siging, kernel_dtype=kernel_dtype, one_launch=one_launch)


def _norm_entry(norm, x):
    """What ``patch_layers`` binds as ``norm.forward``: the fused RMSNorm for CUDA tensors, torch's own otherwise."""
    if x.is_cuda:
        return rms_norm_b200(x, norm.weight, 1e-6 if norm.eps is None else norm.eps)
    return torch.nn.RMSNorm.forward(norm, x)


class _BranchModule(torch.nn.Module):
    """The sub-modules and the parameter ``mlstm_branch_b200`` reads, re-registered (shared, not copied) under one
    parent so that ``torch.cuda.make_graphed_callables`` sees exactly the parameters of the branch."""

    def __init__(self, layer, siging, kernel_dtype, one_launch, amp_dtype):
        super().__init__()
        for name in ("proj_up", "conv", "qk_proj", "v_proj", "mlstm_cell", "proj_down"):
            self.add_module(name, getattr(layer, name))
        self.learnable_skip = layer.learnable_skip
        self.direction = getattr(layer, "direction", None)
        self._cfg = (siging, kernel_dtype, one_launch, amp_dtype)

    def forward(self, x):
        import contextlib

        siging, kernel_dtype, one_launch, amp_dtype = self._cfg
        # the caller's autocast state, re-entered WITHOUT the weight-cast cache: inside a graph every replay must
        # re-round the current fp32 weights (a cached fp16 copy would freeze them at their capture-time values)
        ctx = (torch.autocast("cuda", dtype=amp_dtype, cache_enabled=False) if amp_dtype is not None
               else contextlib.nullcontext())
        with ctx:
            return mlstm_branch_b200(self, x, siging=siging, kernel_dtype=kernel_dtype, one_launch=one_launch)


class _LayerModule(torch.nn.Module):
    """A whole ViLLayer (vision_lstm2.py:331-341: x + mlstm_branch(norm(x)), then + ffn(ffn_norm(.))) under one parent for
    ``torch.cuda.make_graphed_callables``; runs the layer's OWN class forward, so whatever is bound on the instance
    (the fused branch, the fused RMSNorms) is what gets captured."""

    def __init__(self, layer, amp_dtype):
        super().__init__()
        self.add_module("layer", layer)
        self._amp = amp_dtype

    def forward(self, x):
        import contextlib

        ctx = (torch.autocast("cuda", dtype=self._amp, cache_enabled=False) if self._amp is not None
               else contextlib.nullcontext())
        with ctx:
            return type(self.layer).forward(self.layer, x)


class _Graphed:
    """Training-time CUDA graphs of a callable of one (B, S, C) tensor: one forward and one backward graph per
    (input shape, dtype, autocast dtype), built lazily by ``torch.cuda.make_graphed_callables`` at the first training
    call.  A ViLLayer is ~70 kernel launches forward + backward and ~3 ms of host time in eager PyTorch whatever its
    size; at the models' S = 100 / 400 stages that is several times its GPU time (0.5 / 0.9 ms for the mLSTM branch at 32
    images), and with 20 layers per step the host, not the GPU, bounds a training step.  The graphs run the same
    kernels on the same (live) parameters and are bit-identical to the eager code, step after optimizer step
    (tests/test_cell_gpu.py) -- the module is rebuilt with the autocast weight-cast cache off, so every replay
    re-rounds the current fp32 weights.  Calls WITHOUT gradients (inference, the first pass of a checkpointed block)
    replay a forward-only graph captured the same way: static input copy in, clone of the static output out (a
    batch-1 forward of base192 is 20 layers x ~0.6 ms of host time around ~0.1 ms of GPU work).  Calls on the CPU, in a
    multi-process job, during someone else's capture, with stochastic depth active (its batch selection is data
    dependent) or with more than ``max_tokens`` tokens (GPU-bound anyway, and their activations would stay resident
    in the graph's private pool) run eagerly.  One caller at a time per model: a graph owns its static buffers, so two
    threads driving the SAME patched model concurrently must not both use graphs (separate model copies are fine)."""

    def __init__(self, layer, max_tokens=65536, max_graphs=6):
        self.layer = layer
        self.max_tokens, self.max_graphs = max_tokens, max_graphs
        self._graphs = {}

    def __getstate__(self):  # graphs are not picklable / copyable: a copied or loaded model rebuilds them lazily
        d = self.__dict__.copy()
        d["_graphs"] = {}
        return d

    def _eager(self, x):
        raise NotImplementedError

    def _module(self, amp):
        raise NotImplementedError

    def _graphable(self, x) -> bool:
        if torch.compiler.is_compiling():  # torch.compile traces the eager layer (its ops are graph nodes)
            return False
        if (torch.distributed.is_available() and torch.distributed.is_initialized()
                and torch.distributed.get_world_size() > 1):
            # single-process training only: a capture started lazily inside DDP's forward is invalidated by the
            # process group's watchdog thread (global capture mode), and make_graphed_callables wants to run
            # before the DDP wrapper exists (measured: cudaErrorStreamCaptureInvalidated at world size 2)
            return False
        return (x.is_cuda and x.dim() == 3 and x.shape[0] * x.shape[1] <= self.max_tokens
                and not torch.cuda.is_current_stream_capturing())

    def _capture_forward(self, mod, x):
        """Forward-only graph: (graph, static input, static output)."""
        static_in = x.detach().clone()
        side = torch.cuda.Stream(device=x.device)
        side.wait_stream(torch.cuda.current_stream(x.device))
        with torch.no_grad(), torch.autocast("cuda", enabled=False), torch.cuda.stream(side):
            for _ in range(2):  # warm-up outside the capture: plans, tensor maps, cuDNN / cuBLAS workspaces
                mod(static_in)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                static_out = mod(static_in)
        torch.cuda.current_stream(x.device).wait_stream(side)
        return g, static_in, static_out

    @staticmethod
    def _saved_tensor_hooks_active() -> bool:
        """Someone (non-reentrant activation checkpointing, CPU offload) is intercepting what autograd saves: the
        activations of a graph live in its private pool and must not be routed through such hooks."""
        top = getattr(torch._C._autograd, "_top_saved_tensors_default_hooks", None)
        try:
            return top is not None and top(True) is not None
        except Exception:  # noqa: BLE001 -- private API: when in doubt, stay eager
            return True

    def __call__(self, x):
        if not self._graphable(x):
            return self._eager(x)
        train = torch.is_grad_enabled() and x.requires_grad
        if train and self._saved_tensor_hooks_active():
            return self._eager(x)
        if not train and torch.is_grad_enabled() and any(p.requires_grad for p in self.layer.parameters()):
            return self._eager(x)  # gradients w.r.t. the parameters only: rare, not worth a third kind of graph
        amp = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else None
        key = (tuple(x.shape), x.dtype, amp, x.device.index, self.layer.training, train)
        g = self._graphs.get(key)
        if g is None:
            # never build from inside a running backward pass (the re-computation of a checkpointed block,
            # vision_lstm2.py:1071-1078, calls the layer there): that call stays eager
            if len(self._graphs) >= self.max_graphs or torch._C._current_graph_task_id() != -1:
                return self._eager(x)
            mod = self._module(amp)
            mod.train(self.layer.training)
            if train:
                sample = x.detach().clone().requires_grad_(True)
                with torch.autocast("cuda", enabled=False):  # (make_graphed_callables refuses a caching autocast)
                    g = torch.cuda.make_graphed_callables(mod, (sample,), allow_unused_input=True)
            else:
                g = self._capture_forward(mod, x)
            self._graphs[key] = g
        if train:
            return g(x)
        graph, static_in, static_out = g
        static_in.copy_(x)
        graph.replay()
        return static_out.clone()


class _GraphedBranch(_Graphed):
    """``layer.mlstm_branch`` as CUDA graphs (layers without the ViLLayer forward around the branch)."""

    def __init__(self, layer, siging, kernel_dtype, one_launch, **kw):
        super().__init__(layer, **kw)
        self.cfg = (siging, kernel_dtype, one_launch)

    def _eager(self, x):
        siging, kernel_dtype, one_launch = self.cfg
        return mlstm_branch_b200(self.layer, x, siging=siging, kernel_dtype=kernel_dtype, one_launch=one_launch)

    def _module(self, amp):
        return _BranchModule(self.layer, *self.cfg, amp)


class _GraphedLayer(_Graphed):
    """``layer.forward`` of a whole ViLLayer as CUDA graphs: both residual branches, their RMSNorms and the adds."""

    def _eager(self, x):
        return type(self.layer).forward(self.layer, x)

    def _module(self, amp):
        return _LayerModule(self.layer, amp)

    def _graphable(self, x) -> bool:
        dp = getattr(self.layer, "drop_path", None)
        stochastic = dp is not None and self.layer.training and float(getattr(dp, "drop_prob", 0.0)) > 0.0
        return not stochastic and super()._graphable(x)


def patch_layers(model: torch.nn.Module, siging=None, kernel_dtype: str = "bfloat16", one_launch: str = "auto",
                 graphs: bool = False) -> int:
    """Rebind ``mlstm_branch`` of every ViLLayer-shaped module (``proj_up``, ``qk_proj``, ``v_proj``, ``mlstm_cell``,
    ``learnable_skip``, ``proj_down``; vision_lstm2.py:218-290) whose head geometry the fused output kernel covers to
    ``mlstm_branch_b200``.  Parameters and state-dict keys are untouched.  Returns the number of layers rebound.
    ``siging=None`` keeps the gate function of each layer's cell (sigmoid input gate iff the cell's CUDA backend is
    a ``*siging*`` kernel, as in the reference model); True / False force it.

    The overrides are ``functools.partial`` objects over module-level functions, so a patched model (or its EMA
    copy) survives ``copy.deepcopy`` and the whole-module ``torch.save`` / ``torch.load`` the reference trainer
    uses for last.pt / best.pt (ultralytics/engine/trainer.py:517-540): the partial's bound module is pickled as
    part of the same object graph and re-bound to the loaded / copied module.  ``graphs=True`` additionally makes the
    training forward / backward of every such layer replay as CUDA graphs (``_GraphedLayer`` bound as ``layer.forward``
    for a full ViLLayer, ``_GraphedBranch`` as ``layer.mlstm_branch`` otherwise; see ``_Graphed``)."""
    import functools

    n = 0
    for mod in model.modules():
        cell = getattr(mod, "mlstm_cell", None)
        if cell is None or not all(hasattr(mod, a) for a in ("proj_up", "qk_proj", "v_proj", "learnable_skip", "proj_down")):
            continue
        if not cellout_supported(cell.num_heads, cell.dim // cell.num_heads):
            continue
        sig = _cell_uses_siging(cell) if siging is None else bool(siging)
        whole_layer = graphs and all(hasattr(mod, a) for a in ("norm", "ffn_norm", "ffn", "drop_path"))
        if graphs and not whole_layer:
            mod.mlstm_branch = _GraphedBranch(mod, sig, kernel_dtype, one_launch)
        else:
            mod.mlstm_branch = functools.partial(_branch_entry, mod, siging=sig, kernel_dtype=kernel_dtype, one_launch=one_launch)
        if whole_layer:
            mod.forward = _GraphedLayer(mod)
        for norm in (getattr(mod, "norm", None), getattr(mod, "ffn_norm", None)):  # the RMSNorms in front of the branches
            if (isinstance(norm, torch.nn.RMSNorm) and len(norm.normalized_shape) == 1
                    and norm.normalized_shape[0] in RMSNORM_DIMS):
                norm.forward = functools.partial(_norm_entry, norm)
        n += 1
    return n
