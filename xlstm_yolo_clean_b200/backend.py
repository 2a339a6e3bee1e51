"""Host side of the B200 mLSTM chunkwise backend (Python/PyTorch above the C-ABI).

Mirrors the reference's operator interface for this path so it is a drop-in:

  * ``mlstm_chunkwise__b200`` has the signature, return convention, dtype rule and error
    behaviour of ``mlstm_chunkwise__native_custbw`` (mlstm_kernels/torch/chunkwise/native/fwbw.py:228-263);
  * ``mlstm_chunkwise_fw`` / ``mlstm_chunkwise_bw`` correspond to native/fw.py:224-318 and
    native/bw.py:206-348 and are thin wrappers over the two C-ABI calls;
  * ``register`` / ``patch_model`` hook it into mlstm_kernels.torch.chunkwise.registry and
    ``MatrixLSTMCell`` (ultralytics/nn/modules/vision_lstm/vision_lstm2.py:623-770).

PyTorch is used for device memory, streams and autograd plumbing only.  There is no CPU or
eager fallback: CPU tensors or a missing library raise.
"""
from __future__ import annotations

import ctypes as C
import math
import threading
from typing import Optional

import torch
from torch.amp import custom_bwd, custom_fwd

from . import _cabi

KERNEL_NAME = "b200"  # registry key -> "chunkwise--b200"

_DTYPES = {torch.float32: _cabi.F32, torch.bfloat16: _cabi.BF16, torch.float16: _cabi.F16}
_default_impl = _cabi.IMPL_AUTO
_last_launches = 0


def set_default_impl(name: str) -> None:
    """'auto' | 'exact' (fp32 FFMA kernels) | 'tensor' (tcgen05 kernels, error if unsupported)."""
    global _default_impl
    _default_impl = {"auto": _cabi.IMPL_AUTO, "exact": _cabi.IMPL_EXACT, "tensor": _cabi.IMPL_TENSOR}[name]


def last_launch_count() -> int:
    """Kernels launched by the most recent forward or backward call on this thread."""
    return _cabi.load_library().mlstm_b200_last_launch_count()


def _tensor(t: Optional[torch.Tensor]) -> _cabi.Tensor:
    out = _cabi.Tensor()
    if t is None:
        out.ptr = None
        return out
    out.ptr = t.data_ptr()
    st = t.stride()
    out.stride[:len(st)] = st
    return out


class _on_device:
    """``torch.cuda.device(dev)`` only when ``dev`` is not already current (the common case costs nothing)."""

    __slots__ = ("ctx",)

    def __init__(self, dev):
        self.ctx = None if torch.cuda.current_device() == dev.index else torch.cuda.device(dev)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *a):
        if self.ctx is not None:
            self.ctx.__exit__(*a)


def _siging_mode(siging, normalize=True) -> int:
    """``mlstm_b200_shape::siging``: 0 exp input gate, 1 sigmoid input gate, 2 sigmoid input gate without the
    normaliser (``normalize=False``, h = q C + sum_s P_ts v_s).  The exp-gate variant always normalises."""
    if not normalize:
        if not siging:
            raise ValueError("normalize=False exists for the sigmoid input gate only (pass siging=True)")
        return 2
    return 1 if siging else 0


def _siging_flags(mode: int) -> tuple[bool, bool]:
    """(siging, normalize) of a C-ABI mode: the inverse of ``_siging_mode``."""
    return mode != 0, mode != 2


_16BIT = (torch.float16, torch.bfloat16)


def _grad_dtype(kernel_dtype, caller_dtype, tensor_route: bool):
    """The dtype the backward writes freshly allocated gradients in: the caller's dtype (``caller_dtype``, None when
    the caller has no single one) where the tensor-core route rounds its fp32 accumulators straight to it
    (``shape.grad_dtype``: the two 16-bit dtypes), else the kernel dtype (autograd casts the gradients afterwards)."""
    if (caller_dtype is None or caller_dtype is kernel_dtype or not tensor_route or caller_dtype not in _16BIT
            or kernel_dtype not in _16BIT):
        return kernel_dtype
    return caller_dtype


def _zero_c_initial(q, v, c_initial, n_initial, m_initial):
    """``c_initial``, or a zero C when only n / m_initial are given: the kernels read initial states only with a C."""
    if c_initial is None and (n_initial is not None or m_initial is not None):
        B, NH, S, DK = q.shape
        return torch.zeros(B, NH, DK, v.shape[-1], device=q.device)
    return c_initial


def _nm_ptrs(nm):
    """n_out / m_out pointers for the backward from the forward's nm = [n_out, m_out] (2, B, NH, S) fp32, which must be
    contiguous (as the forward allocates it)."""
    nmp = nm.data_ptr()
    return nmp, nmp + nm.stride(0) * 4


def _shape(q, v, chunk_size, eps, impl, qk_scale=None, reverse=False, siging=0, gate_soft_cap=0.0) -> _cabi.Shape:
    B, NH, S, DK = q.shape
    s = _cabi.Shape()
    s.B, s.NH, s.S, s.DHQK, s.DHHV = B, NH, S, DK, v.shape[-1]
    s.chunk_size = int(chunk_size)
    s.dtype = _DTYPES[q.dtype]
    s.impl = _default_impl if impl is None else impl
    s.reverse = 1 if reverse else 0
    s.siging = int(siging)  # _siging_mode
    s.eps = float(eps)
    s.qk_scale = -1.0 if qk_scale is None else float(qk_scale)
    s.gate_soft_cap = float(gate_soft_cap or 0.0)
    return s


def tensor_path_supported(B, NH, S, DK, DV, dtype=torch.bfloat16, chunk_size=64) -> bool:
    s = _cabi.Shape()
    s.B, s.NH, s.S, s.DHQK, s.DHHV, s.chunk_size, s.dtype = B, NH, S, DK, DV, chunk_size, _DTYPES[dtype]
    return bool(_cabi.load_library().mlstm_b200_tensor_path_supported(C.byref(s)))


def _check_inputs(q, k, v, i, f):
    for name, t in (("q", q), ("k", k), ("v", v), ("i", i), ("f", f)):
        if not t.is_cuda:
            raise RuntimeError(f"mlstm_chunkwise__b200: {name} is on {t.device}; this backend has no CPU path")
    if q.dtype not in _DTYPES:
        raise RuntimeError(f"unsupported dtype {q.dtype}")
    B, NH, S, DK = q.shape
    assert k.shape == (B, NH, S, DK), f"k has wrong shape {tuple(k.shape)}"
    assert v.shape[:3] == (B, NH, S), f"v has wrong shape {tuple(v.shape)}"
    assert i.shape == (B, NH, S) and f.shape == (B, NH, S), "i / f must be (B, NH, S)"


def _state_f32(t, shape):
    if t is None:
        return None
    return t.detach().to(torch.float32).reshape(shape).contiguous()


# ------------------------------------------------------------------------------------------------------------------
# Call plans.  A YOLO-ViL training step makes ~90 forward / backward calls of a handful of distinct (shape, strides)
# signatures and is launch-bound on the host, so everything that does not change between two calls of one signature --
# validation, the C-ABI shape / stride structs, scratch sizes, the choice between handing the views to the kernels
# as they are or copying them -- is done once and kept in a per-thread plan (forward runs on the caller's thread,
# backward on an autograd thread, checkpoint recompute re-enters: SURVEY.md section 8b "Threading"; the structs are
# mutated per call, hence thread-local).  Per call: output allocation, ~10 pointer stores, one ctypes call.
# ------------------------------------------------------------------------------------------------------------------
_tls = threading.local()
_raw_stream = torch._C._cuda_getCurrentRawStream


_MAX_PLANS = 1024


def _plans() -> dict:
    """Per-thread call plans (argument structs with everything but the pointers filled in), keyed by the call's
    signature.  A training loop cycles through a few dozen signatures; a caller with ever-changing shapes (variable
    sequence lengths at inference) would otherwise grow the table without bound, so it is simply dropped when full."""
    d = getattr(_tls, "plans", None)
    if d is None:
        d = _tls.plans = {}
    elif len(d) >= _MAX_PLANS:
        d.clear()
    return d


def _tma_strides_ok(t: torch.Tensor) -> bool:
    """What a TMA tensor map needs from a (B, NH, S, D) 16-bit view: unit innermost stride, the other strides
    multiples of 8 elements (16 bytes).  Broadcast (stride 0) dimensions would pass the test but make overlapping
    output rows, so they are copied too."""
    st = t.stride()
    return st[3] == 1 and all(x % 8 == 0 and x > 0 for x in st[:3])


def _tensor_route(lib, shape) -> bool:
    return shape.impl != _cabi.IMPL_EXACT and bool(lib.mlstm_b200_tensor_path_supported(C.byref(shape)))


def _fix_views(tensor_route: bool, ts):
    """The kernels take any batch / head / token strides; what they cannot take is copied here, like the reference's
    @contiguous decorator does for every argument (mlstm_kernels/torch/utils.py:30-42): a non-unit innermost stride
    always, and on the tensor-core route strides that are not multiples of 16 bytes or a base pointer that is not
    16-byte aligned (sliced / offset views)."""
    out = []
    for t in ts:
        if t.stride(-1) != 1 or (tensor_route and t.dim() == 4 and (not _tma_strides_ok(t) or t.data_ptr() & 15)):
            t = t.contiguous()
            if t.data_ptr() & 15:  # a contiguous view at an odd offset of its storage
                t = t.clone()
        out.append(t)
    return out


class _FwPlan:
    __slots__ = ("args", "ref", "ws_bytes", "st_bytes", "tensor_route", "h_shape", "nm_shape", "states", "epi")


class FwEpilogue:
    """Arguments of the fused cell-output epilogue (include/mlstm_b200.h, mlstm_b200_fw_epilogue): ``y`` (out) and ``x``
    (optional skip input) are (B, NH, S, D) VIEWS of 16-bit tensors (e.g. of a (B, S, NH*D) buffer), ``weight`` / ``bias`` /
    ``skip`` contiguous fp32 (NH*D) or None; ``want_h``: also write the un-normalised h (training)."""

    __slots__ = ("y", "x", "weight", "bias", "skip", "eps", "want_h")

    def __init__(self, y, x, weight, bias, skip, eps, want_h):
        self.y, self.x, self.weight, self.bias, self.skip, self.eps, self.want_h = y, x, weight, bias, skip, float(eps), bool(want_h)


class _BwPlan:
    __slots__ = ("args", "ref", "ws_bytes", "tensor_route", "gshape_qk", "gshape_v", "gshape_g")


def _ws_tensor(nbytes: int, dev):
    """Scratch for a call.  The tensor-core forward needs none and its backward only when it has to recompute the
    states; those calls share one tiny per-device buffer instead of allocating 256 bytes each."""
    if nbytes <= 256:
        cache = getattr(_tls, "tiny_ws", None)
        if cache is None:
            cache = _tls.tiny_ws = {}
        t = cache.get(dev.index)
        if t is None:
            t = cache[dev.index] = torch.empty(256, dtype=torch.uint8, device=dev)
        return t
    return torch.empty(nbytes, dtype=torch.uint8, device=dev)


def _fw_launch(q, k, v, i, f, c0, n0, m0, qk_scale, return_last_states, chunk_size, eps, impl, save_states, reverse, siging,
               soft_cap=0.0, epi: Optional[FwEpilogue] = None):
    """Returns h, nm (2, B, NH, S) fp32 = [n_out, m_out], last-or-None, c_states-or-None.  With ``epi`` the kernel writes
    epi.y (fused LayerNorm + skip epilogue) and h is None unless epi.want_h.  ``siging``: the C-ABI mode, see
    ``_siging_mode`` (a bool is mode 0 / 1)."""
    impl = _default_impl if impl is None else impl
    dt = q.dtype
    if i.dtype is not dt:
        i = i.to(dt)
    if f.dtype is not dt:
        f = f.to(dt)
    if k.dtype is not dt:
        k = k.to(dt)
    if v.dtype is not dt:
        v = v.to(dt)
    dev = q.device
    key = (0, q.shape, v.shape[3], dt, q.stride(), k.stride(), v.stride(), i.stride(), f.stride(), chunk_size, eps, impl,
           qk_scale, reverse, siging, c0 is not None, return_last_states, save_states, dev.index, soft_cap,
           None if epi is None else (epi.y.stride(), epi.y.dtype, None if epi.x is None else epi.x.stride(), epi.want_h,
                                     epi.weight is None, epi.bias is None, epi.skip is None, epi.eps))
    plans = _plans()
    plan = plans.get(key)
    lib = _cabi.load_library()
    if plan is None:
        _check_inputs(q, k, v, i, f)
        B, NH, S, DK = q.shape
        assert S % chunk_size == 0, f"Sequence length {S} is not divisible by chunk size {chunk_size}."
        a = _cabi.FwArgs()
        a.shape = _shape(q, v, chunk_size, eps, impl, qk_scale, reverse, siging, soft_cap)
        plan = _FwPlan()
        plan.tensor_route = _tensor_route(lib, a.shape)
        if soft_cap and not plan.tensor_route:
            raise RuntimeError("gate_soft_cap is applied in-kernel on the tensor-core route only; cap the gates first")
        fixed = _fix_views(plan.tensor_route, (q, k, v))
        if any(x is not y for x, y in zip(fixed, (q, k, v))):  # a signature that needs copies: plan on the copies
            return _fw_launch(*fixed, i, f, c0, n0, m0, qk_scale, return_last_states, chunk_size, eps, impl, save_states,
                              reverse, siging, soft_cap, epi)
        plan.ws_bytes = lib.mlstm_b200_workspace_bytes(C.byref(a.shape), 0)
        plan.st_bytes = lib.mlstm_b200_states_bytes(C.byref(a.shape)) if save_states else 0
        plan.h_shape, plan.nm_shape = (B, NH, S, v.shape[3]), (2, B, NH, S)
        plan.states = ((B, NH, DK, v.shape[3]), (B, NH, DK), (B, NH))
        for name, t in (("q", q), ("k", k), ("v", v), ("i", i), ("f", f)):
            getattr(a, name).stride[:t.dim()] = t.stride()
        a.h.stride[:4] = (NH * S * v.shape[3], S * v.shape[3], v.shape[3], 1)
        a.workspace_bytes = max(plan.ws_bytes, 256)
        plan.epi = None
        if epi is not None:
            if not plan.tensor_route:
                raise RuntimeError("the fused cell-output epilogue exists on the tensor-core route only")
            assert epi.y.shape == plan.h_shape and epi.y.dtype in (torch.float16, torch.bfloat16)
            assert epi.x is None or (epi.x.shape == plan.h_shape and epi.x.dtype == epi.y.dtype)
            if not _tma_strides_ok(epi.y) or (epi.x is not None and not _tma_strides_ok(epi.x)):
                raise RuntimeError("fused epilogue: y / x need a unit innermost stride and 16-byte-multiple strides")
            e = _cabi.FwEpilogue()
            e.y.stride[:4] = epi.y.stride()
            if epi.x is not None:
                e.x.stride[:4] = epi.x.stride()
            e.eps, e.xy_dtype = epi.eps, _DTYPES[epi.y.dtype]
            plan.epi = e
            a.epilogue = C.pointer(e)
        plan.args, plan.ref = a, C.byref(a)
        plans[key] = plan
    elif plan.tensor_route and (q.data_ptr() | k.data_ptr() | v.data_ptr()) & 15:  # offset views of this signature
        q, k, v = _fix_views(True, (q, k, v))
    a = plan.args
    if torch._C._cuda_getDevice() != dev.index:
        with torch.cuda.device(dev):
            return _fw_launch(q, k, v, i, f, c0, n0, m0, qk_scale, return_last_states, chunk_size, eps, impl, save_states,
                              reverse, siging, soft_cap, epi)
    h = torch.empty(plan.h_shape, dtype=dt, device=dev) if (epi is None or epi.want_h) else None
    nm = torch.empty(plan.nm_shape, dtype=torch.float32, device=dev)
    c_states = torch.empty(plan.st_bytes, dtype=torch.uint8, device=dev) if plan.st_bytes else None
    ws = _ws_tensor(plan.ws_bytes, dev)
    last = None
    if c0 is not None:
        sc, sn, sm = plan.states
        c0, n0, m0 = _state_f32(c0, sc), _state_f32(n0, sn), _state_f32(m0, sm)
        n0 = torch.zeros(sn, device=dev) if n0 is None else n0
        m0 = torch.zeros(sm, device=dev) if m0 is None else m0
        a.c_initial, a.n_initial, a.m_initial = c0.data_ptr(), n0.data_ptr(), m0.data_ptr()
    if return_last_states:
        sc, sn, sm = plan.states
        last = (torch.empty(sc, dtype=torch.float32, device=dev), torch.empty(sn, dtype=torch.float32, device=dev),
                torch.empty(sm + (1,), dtype=torch.float32, device=dev))
        a.c_last, a.n_last, a.m_last = last[0].data_ptr(), last[1].data_ptr(), last[2].data_ptr()
    a.q.ptr, a.k.ptr, a.v.ptr, a.i.ptr, a.f.ptr = q.data_ptr(), k.data_ptr(), v.data_ptr(), i.data_ptr(), f.data_ptr()
    a.h.ptr = h.data_ptr() if h is not None else None
    if epi is not None:
        e = plan.epi
        if (epi.y.data_ptr() | (0 if epi.x is None else epi.x.data_ptr())) & 15:
            raise RuntimeError("fused epilogue: y / x must be 16-byte aligned")
        e.y.ptr = epi.y.data_ptr()
        e.x.ptr = None if epi.x is None else epi.x.data_ptr()
        e.weight = None if epi.weight is None else epi.weight.data_ptr()
        e.bias = None if epi.bias is None else epi.bias.data_ptr()
        e.skip = None if epi.skip is None else epi.skip.data_ptr()
    nmp = nm.data_ptr()
    a.n_out, a.m_out = nmp, nmp + nm.stride(0) * 4
    a.c_states = c_states.data_ptr() if c_states is not None else None
    a.workspace = ws.data_ptr()
    st = lib.mlstm_b200_chunkwise_fw(plan.ref, _raw_stream(dev.index))
    if st:
        _cabi.check(st, "mlstm_b200_chunkwise_fw")
    return h, nm, last, c_states


def _is_dense(x) -> bool:
    """A permutation of a contiguous buffer: every element of the storage range is addressed exactly once."""
    if x.is_contiguous():
        return True
    expected = 1
    for st, sz in sorted(zip(x.stride(), x.shape)):
        if sz == 1:
            continue
        if st != expected:
            return False
        expected *= sz
    return True


def convert16(x: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """``x.to(dtype)`` for fp16 <-> bf16 CUDA tensors as one streaming pass (C-ABI ``mlstm_b200_convert16``): the
    re-rounding the reference kernels apply to their inputs under autocast (native/fwbw.py:37), bit-identical to torch's,
    at twice its rate.  Dense tensors only (any permutation of a contiguous buffer keeps its strides); everything else
    goes through torch."""
    if x.dtype is dtype:
        return x
    if torch.compiler.is_compiling():
        return _ops.convert16(x, dtype)
    if (not x.is_cuda or {x.dtype, dtype} != {torch.float16, torch.bfloat16} or x.numel() == 0
            or not _is_dense(x)):
        return x.to(dtype)
    y = torch.empty_like(x, dtype=dtype)  # preserve_format: same strides for a dense tensor
    if y.stride() != x.stride():
        return x.to(dtype)
    dev = x.device
    if torch._C._cuda_getDevice() != dev.index:
        with torch.cuda.device(dev):
            return convert16(x, dtype)
    st = _cabi.load_library().mlstm_b200_convert16(x.data_ptr(), y.data_ptr(), x.numel(), _DTYPES[x.dtype], _DTYPES[dtype],
                                                  _raw_stream(dev.index))
    if st:
        _cabi.check(st, "mlstm_b200_convert16")
    return y


def mlstm_chunkwise_fw(q, k, v, i, f, c_initial=None, n_initial=None, m_initial=None, qk_scale=None,
                       return_last_states=False, chunk_size=64, eps=1e-6, impl=None, save_states=True, reverse=False, siging=False,
                       gate_soft_cap=0.0, normalize=True):
    """C-ABI forward.  Returns h, n_out, m_out, last_states-or-None (fp32), c_states-or-None.

    ``normalize=False`` (sigmoid input gate only, ``ValueError`` otherwise): h is the numerator q C + sum_s P_ts v_s,
    without the division by max(|n|, 1) + eps; n_out / m_out are written as with the normaliser, and the last states
    are the same.

    ``gate_soft_cap`` > 0: ``i`` / ``f`` are gate pre-activations and the kernel applies ``cap * tanh(x / cap)``
    (MatrixLSTMCell.soft_cap, vision_lstm2.py:714-715) while it scans them (tensor-core route only).

    ``c_states`` is the opaque per-tile state buffer the tensor-core backward consumes (the
    reference's return_all_states mode, native/fwbw.py:73-101); None when the kernels recompute."""
    mode = _siging_mode(siging, normalize)
    c_initial = _zero_c_initial(q, v, c_initial, n_initial, m_initial)
    launch = _ops.fw_launch if torch.compiler.is_compiling() else _fw_launch
    h, nm, last, c_states = launch(q, k, v, i, f, c_initial, n_initial, m_initial, qk_scale, bool(return_last_states),
                                   int(chunk_size), float(eps), impl, bool(save_states), bool(reverse), mode,
                                   float(gate_soft_cap or 0.0))
    return h, nm[0], nm[1], last, c_states


def _bw_launch(q, k, v, i, f, n_ptr, m_ptr, dh, c0, n0, m0, dcl, qk_scale, chunk_size, eps, impl, want_dc_initial, c_states,
               reverse, siging, out, soft_cap=0.0, grad_dtype=None):
    """``out``: caller-owned (dq, dk, dv, di, df).  Their dtype (or ``grad_dtype`` when the gradients are allocated here)
    may be the OTHER 16-bit dtype than the kernel's: the tensor-core backward then rounds its fp32 accumulators straight
    to it (``shape.grad_dtype``) -- a bf16 kernel under fp16 autocast needs no cast pass over the gradients."""
    impl = _default_impl if impl is None else impl
    dt = q.dtype
    gdt = out[0].dtype if out is not None else (grad_dtype or dt)
    if dh.dtype is not dt:
        dh = dh.to(dt)
    if i.dtype is not dt:
        i = i.to(dt)
    if f.dtype is not dt:
        f = f.to(dt)
    dev = q.device
    key = (1, q.shape, v.shape[3], dt, q.stride(), k.stride(), v.stride(), i.stride(), f.stride(), dh.stride(), chunk_size, eps,
           impl, qk_scale, reverse, siging, c0 is not None, want_dc_initial, c_states is not None, dev.index,
           None if out is None else tuple(t.stride() for t in out), soft_cap, gdt)
    plans = _plans()
    plan = plans.get(key)
    lib = _cabi.load_library()
    if plan is None:
        _check_inputs(q, k, v, i, f)
        B, NH, S, DK = q.shape
        DV = v.shape[3]
        a = _cabi.BwArgs()
        a.shape = _shape(q, v, chunk_size, eps, impl, qk_scale, reverse, siging, soft_cap)
        plan = _BwPlan()
        plan.tensor_route = _tensor_route(lib, a.shape)
        if gdt is not dt:
            if out is None and _grad_dtype(dt, gdt, plan.tensor_route) is dt:
                return _bw_launch(q, k, v, i, f, n_ptr, m_ptr, dh, c0, n0, m0, dcl, qk_scale, chunk_size, eps, impl,
                                  want_dc_initial, c_states, reverse, siging, None, soft_cap, None)
            if not plan.tensor_route or gdt not in (torch.float16, torch.bfloat16):
                raise RuntimeError(f"gradients in {gdt} from a {dt} kernel: tensor-core route and 16-bit dtypes only")
            a.shape.grad_dtype = _DTYPES[gdt]
        fixed = _fix_views(plan.tensor_route, (q, k, v, dh))
        if any(x is not y for x, y in zip(fixed, (q, k, v, dh))):
            return _bw_launch(*fixed[:3], i, f, n_ptr, m_ptr, fixed[3], c0, n0, m0, dcl, qk_scale, chunk_size, eps, impl,
                              want_dc_initial, c_states, reverse, siging, out, soft_cap, grad_dtype)
        if out is not None:
            dq, dk, dv, di, df = out
            assert dq.shape == q.shape and dk.shape == k.shape and dv.shape == v.shape and di.shape == i.shape
            assert all(t.dtype == gdt and t.device == dev for t in out)
            if plan.tensor_route and not all(_tma_strides_ok(t) for t in (dq, dk, dv)):
                raise RuntimeError("caller-provided dq / dk / dv need a unit innermost stride and 16-byte-multiple strides")
            for name, t in zip(("dq", "dk", "dv", "di", "df"), out):
                getattr(a, name).stride[:t.dim()] = t.stride()
        else:
            a.dq.stride[:4] = a.dk.stride[:4] = (NH * S * DK, S * DK, DK, 1)
            a.dv.stride[:4] = (NH * S * DV, S * DV, DV, 1)
            a.di.stride[:3] = a.df.stride[:3] = (NH * S, S, 1)
        # the tensor-core route only needs scratch to recompute the states (or for the block problems of head dim 128
        # and of rectangular heads)
        plan.ws_bytes = lib.mlstm_b200_workspace_bytes(C.byref(a.shape), 1)
        if plan.tensor_route and c_states is not None and DK != 128 and DK == DV:
            plan.ws_bytes = 0
        plan.gshape_qk, plan.gshape_v, plan.gshape_g = (B, NH, S, DK), (B, NH, S, DV), (B, NH, S)
        for name, t in (("q", q), ("k", k), ("v", v), ("i", i), ("f", f), ("dh", dh)):
            getattr(a, name).stride[:t.dim()] = t.stride()
        a.workspace_bytes = max(plan.ws_bytes, 256)
        plan.args, plan.ref = a, C.byref(a)
        plans[key] = plan
    elif plan.tensor_route and (q.data_ptr() | k.data_ptr() | v.data_ptr() | dh.data_ptr()) & 15:
        q, k, v, dh = _fix_views(True, (q, k, v, dh))
    a = plan.args
    if torch._C._cuda_getDevice() != dev.index:
        with torch.cuda.device(dev):
            return _bw_launch(q, k, v, i, f, n_ptr, m_ptr, dh, c0, n0, m0, dcl, qk_scale, chunk_size, eps, impl,
                              want_dc_initial, c_states, reverse, siging, out, soft_cap, grad_dtype)
    if out is not None:
        dq, dk, dv, di, df = out
        if plan.tensor_route and (dq.data_ptr() | dk.data_ptr() | dv.data_ptr()) & 15:
            raise RuntimeError("caller-provided dq / dk / dv must be 16-byte aligned")
    else:
        dq = torch.empty(plan.gshape_qk, dtype=gdt, device=dev)
        dk = torch.empty(plan.gshape_qk, dtype=gdt, device=dev)
        dv = torch.empty(plan.gshape_v, dtype=gdt, device=dev)
        di = torch.empty(plan.gshape_g, dtype=gdt, device=dev)
        df = torch.empty(plan.gshape_g, dtype=gdt, device=dev)
    ws = _ws_tensor(plan.ws_bytes, dev)
    dc0 = None
    if c0 is not None:
        B, NH, S, DK = q.shape
        DV = v.shape[3]
        c0, n0, m0 = _state_f32(c0, (B, NH, DK, DV)), _state_f32(n0, (B, NH, DK)), _state_f32(m0, (B, NH))
        n0 = torch.zeros(B, NH, DK, device=dev) if n0 is None else n0
        m0 = torch.zeros(B, NH, device=dev) if m0 is None else m0
        a.c_initial, a.n_initial, a.m_initial = c0.data_ptr(), n0.data_ptr(), m0.data_ptr()
    if want_dc_initial:
        dc0 = torch.empty(q.shape[0], q.shape[1], q.shape[3], v.shape[3], dtype=torch.float32, device=dev)
        a.dc_initial = dc0.data_ptr()
    if dcl is not None:
        dcl = _state_f32(dcl, (q.shape[0], q.shape[1], q.shape[3], v.shape[3]))
    a.dc_last = None if dcl is None else dcl.data_ptr()
    a.q.ptr, a.k.ptr, a.v.ptr, a.i.ptr, a.f.ptr, a.dh.ptr = (q.data_ptr(), k.data_ptr(), v.data_ptr(), i.data_ptr(),
                                                             f.data_ptr(), dh.data_ptr())
    a.dq.ptr, a.dk.ptr, a.dv.ptr, a.di.ptr, a.df.ptr = (dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), di.data_ptr(),
                                                        df.data_ptr())
    a.n_out, a.m_out = n_ptr, m_ptr
    a.c_states = c_states.data_ptr() if c_states is not None else None
    a.workspace = ws.data_ptr()
    st = lib.mlstm_b200_chunkwise_bw(plan.ref, _raw_stream(dev.index))
    if st:
        _cabi.check(st, "mlstm_b200_chunkwise_bw")
    return dq, dk, dv, di, df, dc0


def mlstm_chunkwise_bw(q, k, v, i, f, n_out, m_out, dh, c_initial=None, n_initial=None, m_initial=None,
                       dc_last=None, qk_scale=None, chunk_size=64, eps=1e-6, impl=None, want_dc_initial=False,
                       c_states=None, reverse=False, siging=False, out=None, gate_soft_cap=0.0, grad_dtype=None,
                       normalize=True):
    """C-ABI backward.  Returns dq, dk, dv, di, df, dc_initial-or-None (fp32).

    ``normalize=False`` (sigmoid input gate only, ``ValueError`` otherwise): the backward of the forward's
    ``normalize=False``; dh is not scaled by 1 / (n_out + eps) and ``n_out`` is not read.

    With ``gate_soft_cap`` > 0 (see the forward) di / df are gradients w.r.t. the gate pre-activations.

    ``out`` = (dq, dk, dv, di, df) lets the caller provide the gradient tensors (any batch/head/token strides,
    unit innermost stride for dq/dk/dv), e.g. views into a fused (B, S, 2H) qk gradient.  Their dtype -- or
    ``grad_dtype`` when the gradients are allocated here -- may be the other 16-bit dtype than the kernel's."""
    mode = _siging_mode(siging, normalize)
    c_initial = _zero_c_initial(q, v, c_initial, n_initial, m_initial)
    launch = _ops.bw_launch if torch.compiler.is_compiling() else _chunkwise_bw
    return launch(q, k, v, i, f, n_out, m_out, dh, c_initial, n_initial, m_initial, dc_last, qk_scale, int(chunk_size),
                  float(eps), impl, bool(want_dc_initial), c_states, bool(reverse), mode, out, float(gate_soft_cap or 0.0),
                  grad_dtype)


def _chunkwise_bw(q, k, v, i, f, n_out, m_out, dh, c0, n0, m0, dc_last, qk_scale, chunk_size, eps, impl, want_dc_initial,
                  c_states, reverse, siging, out, soft_cap, grad_dtype):
    """``_bw_launch`` with n_out / m_out as (B, NH, S) fp32 tensors (copied where they are not contiguous)."""
    n_out, m_out = n_out.contiguous(), m_out.contiguous()
    return _bw_launch(q, k, v, i, f, n_out.data_ptr(), m_out.data_ptr(), dh, c0, n0, m0, dc_last, qk_scale, chunk_size, eps,
                      impl, want_dc_initial, c_states, reverse, siging, out, soft_cap, grad_dtype)


def _make_function(autocast_kernel_dtype: torch.dtype):
    class _MlstmChunkwiseB200(torch.autograd.Function):
        """autograd.Function with the contract of _mlstm_chunkwise_fwbw (native/fwbw.py:35-171).  ``siging`` is the
        C-ABI mode of ``_siging_mode`` (0 / 1 / 2)."""

        @staticmethod
        @custom_fwd(device_type="cuda", cast_inputs=autocast_kernel_dtype)
        def forward(ctx, q, k, v, i, f, c_initial, n_initial, m_initial, return_last_states, chunk_size, eps, reverse,
                    siging, grad_dtype=None):
            need_bw = any(ctx.needs_input_grad[:6])
            ctx.grad_dtype = grad_dtype
            h, nm, last, c_states = _fw_launch(q, k, v, i, f, c_initial, n_initial, m_initial, None, return_last_states,
                                               chunk_size, eps, None, need_bw, reverse, siging)
            ctx.save_for_backward(q, k, v, i, f, c_initial, n_initial, m_initial, nm, c_states)
            ctx.chunk_size, ctx.eps, ctx.reverse, ctx.siging = chunk_size, eps, reverse, siging
            if last is None:
                return h, None, None, None
            # native kernels hand states back in the input dtype (native/fw.py:53-62)
            return h, last[0].to(q.dtype), last[1].to(q.dtype), last[2].to(q.dtype)

        @staticmethod
        @custom_bwd(device_type="cuda")
        def backward(ctx, dh, dc_last, dn_last, dm_last):
            q, k, v, i, f, c0, n0, m0, nm, c_states = ctx.saved_tensors
            n_ptr, m_ptr = _nm_ptrs(nm)
            dq, dk, dv, di, df, dc0 = _bw_launch(q, k, v, i, f, n_ptr, m_ptr, dh, c0, n0, m0, dc_last, None,
                                                 ctx.chunk_size, ctx.eps, None, c0 is not None, c_states, ctx.reverse,
                                                 ctx.siging, None, 0.0, ctx.grad_dtype)
            # dn_last / dm_last are ignored and dN/dM_initial are zeros, as in native/bw.py:329-337
            return (dq, dk, dv, di, df,
                    None if c0 is None else dc0.to(c0.dtype),
                    None if n0 is None else torch.zeros_like(n0),
                    None if m0 is None else torch.zeros_like(m0),
                    None, None, None, None, None, None)

    return _MlstmChunkwiseB200


def _caller_grad_dtype(kernel_dtype, *tensors):
    """Under CUDA autocast custom_fwd re-rounds 16-bit inputs to the kernel dtype and autograd casts the gradients back:
    when every differentiable input has the same OTHER 16-bit dtype the backward kernel writes that dtype itself."""
    if not torch.is_autocast_enabled("cuda"):
        return None
    dt = tensors[0].dtype
    if dt is kernel_dtype or dt not in (torch.float16, torch.bfloat16) or kernel_dtype not in (torch.float16, torch.bfloat16):
        return None
    return dt if all(t.dtype is dt for t in tensors) else None


_FUNCTIONS = {dt: _make_function(dt) for dt in (torch.float32, torch.float16, torch.bfloat16)}


def mlstm_chunkwise__b200(
    q: torch.Tensor,
    k: torch.Tensor,
    v: torch.Tensor,
    i: torch.Tensor,
    f: torch.Tensor,
    c_initial: torch.Tensor = None,
    n_initial: torch.Tensor = None,
    m_initial: torch.Tensor = None,
    return_last_states: bool = False,
    eps: float = 1e-6,
    chunk_size: int = 64,
    autocast_kernel_dtype: torch.dtype = torch.bfloat16,
    reverse: bool = False,
    **kwargs,
):
    """Drop-in for ``mlstm_chunkwise__native_custbw`` (native/fwbw.py:228-263).

    ``reverse=True`` (extension) runs the anti-causal scan: the result equals
    ``flip(f(flip(q), flip(k), ...))`` along S -- what ViLLayer obtains with two ``x.flip`` copies for
    its bottom-right direction (vision_lstm2.py:292-312) -- without moving any data.

    Returns h (B, NH, S, DHHV) or (h, (C_last, n_last, m_last)) when ``return_last_states``.
    Extra keyword arguments are ignored like ``native_autograd`` does (fwbw.py:204).
    """
    if autocast_kernel_dtype not in _FUNCTIONS:
        raise ValueError(f"Unsupported kernel dtype {autocast_kernel_dtype}.")
    fn = _FUNCTIONS[autocast_kernel_dtype]
    if torch.compiler.is_compiling():
        fn = _ops.chunkwise_function(autocast_kernel_dtype)
    c_initial = _zero_c_initial(q, v, c_initial, n_initial, m_initial)
    h, c_last, n_last, m_last = fn.apply(q, k, v, i, f, c_initial, n_initial, m_initial, bool(return_last_states),
                                         int(chunk_size), float(eps), bool(reverse), False,
                                         _caller_grad_dtype(autocast_kernel_dtype, q, k, v, i, f))
    if return_last_states:
        return h, (c_last, n_last, m_last)
    return h


def mlstm_siging_chunkwise__b200(
    q: torch.Tensor,
    k: torch.Tensor,
    v: torch.Tensor,
    i: torch.Tensor,
    f: torch.Tensor,
    c_initial: torch.Tensor = None,
    n_initial: torch.Tensor = None,
    return_last_states: bool = False,
    eps: float = 1e-6,
    normalize: bool = True,
    chunk_size: int = 64,
    autocast_kernel_dtype: torch.dtype = torch.bfloat16,
    reverse: bool = False,
    **kwargs,
):
    """Sigmoid-input-gate variant: drop-in for ``mlstm_siging_chunkwise__xl_chunk``
    (mlstm_kernels/torch/chunkwise/triton_xl_chunk_siging/fwbw.py:211-268), the kernel the reference's
    CUDA model path selects (vision_lstm2.py:685-697).  No max state: last states are (C, n).
    ``normalize=False`` drops the normaliser: h = q C + sum_s P_ts v_s, with no division by max(|n|, 1) + eps (n is
    still carried and returned).  The Triton tile-size kwargs are accepted and ignored.
    """
    if autocast_kernel_dtype not in _FUNCTIONS:
        raise ValueError(f"Unsupported kernel dtype {autocast_kernel_dtype}.")
    fn = _FUNCTIONS[autocast_kernel_dtype]
    if torch.compiler.is_compiling():
        fn = _ops.chunkwise_function(autocast_kernel_dtype)
    c_initial = _zero_c_initial(q, v, c_initial, n_initial, None)  # no max state: the kernels start m at 0
    h, c_last, n_last, _ = fn.apply(q, k, v, i, f, c_initial, n_initial, None, bool(return_last_states),
                                    int(chunk_size), float(eps), bool(reverse), _siging_mode(True, normalize),
                                    _caller_grad_dtype(autocast_kernel_dtype, q, k, v, i, f))
    if return_last_states:
        return h, (c_last, n_last)
    return h


def mlstm_recurrent_sequence__b200(q, k, v, i, f, c_initial=None, n_initial=None, m_initial=None,
                                   return_last_states: bool = False, eps: float = 1e-6,
                                   dtype_state: torch.dtype = torch.float32, siging: bool = False, normalize: bool = True,
                                   **kwargs):
    """Token-by-token mLSTM over a whole sequence in ONE launch, state on chip: drop-in for
    ``mlstm_recurrent_sequence__native_fw`` (mlstm_kernels/torch/recurrent/native_sequence.py:133-175; registry name
    ``native_sequence__native``).  q, k (B, NH, S, DHQK), v (B, NH, S, DHHV), i, f (B, NH, S).
    ``siging=True, normalize=False``: the sigmoid-input-gate cell without the normaliser (h = q . C_t), so that a
    ``return_last_states`` prefix of ``mlstm_siging_chunkwise__b200(normalize=False)`` continues here.
    Returns h, or (h, (C, n, m)) with ``return_last_states`` -- the reference's convention; forward only."""
    mode = _siging_mode(siging, normalize)
    if torch.compiler.is_compiling():
        return _ops.recurrent_sequence(q, k, v, i, f, c_initial, n_initial, m_initial, bool(return_last_states), float(eps),
                                       dtype_state, bool(siging), normalize=bool(normalize))
    lib = _cabi.load_library()
    for name, t in (("q", q), ("k", k), ("v", v), ("i", i), ("f", f)):
        if not t.is_cuda:
            raise RuntimeError(f"mlstm_recurrent_sequence__b200: {name} is on {t.device}; this backend has no CPU path")
    B, NH, S, DK = q.shape
    DV = v.shape[-1]
    dt = q.dtype
    if dt not in _DTYPES:
        raise RuntimeError(f"unsupported dtype {dt}")
    q, k, v = (t if t.stride(-1) == 1 else t.contiguous() for t in (q, k.to(dt), v.to(dt)))
    i, f = i.reshape(B, NH, S).to(dt), f.reshape(B, NH, S).to(dt)
    dev = q.device
    with _on_device(dev):
        a = _cabi.RecurrentArgs()
        a.B, a.NH, a.S, a.DHQK, a.DHHV, a.dtype, a.siging, a.eps = B, NH, S, DK, DV, _DTYPES[dt], mode, float(eps)
        h = torch.empty(B, NH, S, DV, dtype=dt, device=dev)
        a.q, a.k, a.v, a.i, a.f, a.h = (_tensor(t) for t in (q, k, v, i, f, h))
        keep = []
        if c_initial is not None:
            c0 = _state_f32(c_initial, (B, NH, DK, DV))
            n0 = _state_f32(n_initial, (B, NH, DK)) if n_initial is not None else torch.zeros(B, NH, DK, device=dev)
            m0 = _state_f32(m_initial, (B, NH)) if m_initial is not None else torch.zeros(B, NH, device=dev)
            keep = [c0, n0, m0]
            a.c_initial, a.n_initial, a.m_initial = c0.data_ptr(), n0.data_ptr(), m0.data_ptr()
        last = None
        if return_last_states:
            last = (torch.empty(B, NH, DK, DV, dtype=torch.float32, device=dev),
                    torch.empty(B, NH, DK, dtype=torch.float32, device=dev),
                    torch.empty(B, NH, 1, dtype=torch.float32, device=dev))
            a.c_last, a.n_last, a.m_last = (t.data_ptr() for t in last)
        st = lib.mlstm_b200_recurrent_sequence(C.byref(a), _raw_stream(dev.index))
        _cabi.check(st, "mlstm_b200_recurrent_sequence")
    if last is None:
        return h
    return h, tuple(t.to(dtype_state) for t in last)


def mlstm_recurrent_step__b200(q, k, v, i, f, c, n, m, eps: float = 1e-6, dtype_state: torch.dtype = torch.float32,
                               siging: bool = False, normalize: bool = True, **kwargs):
    """One recurrent step: drop-in for ``mlstm_recurrent_step__native`` (recurrent/native_step.py:104-132; registry name
    ``native``).  q, k (B, NH, DHQK), v (B, NH, DHHV), i, f (B, NH, 1); states c (B, NH, DHQK, DHHV), n (B, NH, DHQK),
    m (B, NH, 1).  Returns h (B, NH, DHHV), (c_new, n_new, m_new)."""
    h, last = mlstm_recurrent_sequence__b200(q.unsqueeze(2), k.unsqueeze(2), v.unsqueeze(2), i.reshape(*i.shape[:2], 1),
                                             f.reshape(*f.shape[:2], 1), c, n, m, return_last_states=True, eps=eps,
                                             dtype_state=dtype_state, siging=siging, normalize=normalize)
    return h.squeeze(2), last


def register(name: str = KERNEL_NAME) -> str:
    """Insert the kernels into the reference registry (mlstm_kernels/torch/chunkwise/__init__.py:9-15):
    ``<name>`` (exp input gate, max-state stabilised) and ``<name>_siging`` (sigmoid input gate).

    Returns the full kernel name usable as ``mLSTMBackendConfig(chunkwise_kernel=...)``.
    ``mlstm_kernels`` must be importable (it is the reference's package, not part of this repo).
    """
    from mlstm_kernels.torch.chunkwise import registry  # noqa: WPS433 (reference package)

    registry[name] = mlstm_chunkwise__b200
    registry[name + "_siging"] = mlstm_siging_chunkwise__b200
    try:  # the recurrent registries (mlstm_kernels/torch/recurrent/__init__.py:14-25): step_kernel="b200",
        from mlstm_kernels.torch.recurrent import registry_sequence, registry_step  # sequence_kernel="native_sequence__b200"

        registry_step[name] = mlstm_recurrent_step__b200
        registry_sequence["native_sequence__" + name] = mlstm_recurrent_sequence__b200
    except ImportError:  # pragma: no cover
        pass
    return f"chunkwise--{name}"


def _cell_uses_siging(cell) -> bool:
    """True if the cell's current CUDA backend is a sigmoid-input-gate kernel (its ``chunkwise_kernel`` name
    carries ``siging``: ``chunkwise--triton_xl_chunk_siging`` in the reference, vision_lstm2.py:685-697)."""
    cfg = getattr(getattr(cell, "gpu_backend", None), "config", None)
    return "siging" in str(getattr(cfg, "chunkwise_kernel", ""))


def patch_model(model: torch.nn.Module, name: str = KERNEL_NAME, mode: str = "train_with_padding",
                siging: Optional[bool] = None, fused: bool = False, kernel_dtype: str = "bfloat16",
                keep_activations: bool = False, graphs: bool = False) -> int:
    """Point ``gpu_backend`` of every MatrixLSTMCell (vision_lstm2.py:685-697) at the B200 kernel.

    ``siging=None`` (default) keeps the FUNCTION each cell computes on CUDA: a cell whose ``gpu_backend`` is a
    sigmoid-input-gate kernel -- the reference's CUDA default ``chunkwise--triton_xl_chunk_siging`` (sigmoid
    input gate, denominator max(|n|, 1)) -- gets ``chunkwise--b200_siging``, so released weights keep their
    meaning; any other cell gets the exp-gate / max-state kernel.  ``siging=True`` / ``False`` force one variant
    for every cell (``False`` = the function the reference runs on CPU, SURVEY.md finding 6; the parity oracle).
    ``fused=True`` additionally rebinds ``ViLLayer.mlstm_branch`` (vision_lstm2.py:292-312) to
    ``vil.mlstm_branch_b200``: same parameters and function, but the cell's output stage (MultiHeadLayerNorm +
    relayout + learnable skip) runs as one fused CUDA pass each way, the bottom-right direction uses the
    kernel's anti-causal scan instead of two ``x.flip`` copies, and q/k/v are consumed as strided views
    (SURVEY.md section 8(f) #2, #3).

    ``keep_activations=True`` raises ``ViLBlockPair.ckpt_thresh`` (vision_lstm2.py:1030, 1071-1078) so that the
    two S=6400 block pairs stop re-running their forward inside the backward: the reference checkpoints them to
    fit 40-80 GB parts; a B=32 base256 step peaks at ~22 GB of the B200's 180 GB with checkpointing on.
    ``graphs=True`` (with ``fused=True``): the fused branches replay as CUDA graphs in training
    (``vil._GraphedBranch``: a step of the patched model is otherwise bound by the host's launch rate).
    Returns the number of cells patched.
    """
    from mlstm_kernels.torch.backend_module import mLSTMBackend, mLSTMBackendConfig

    if graphs and not fused:
        raise ValueError("graphs=True replays the FUSED layers as CUDA graphs: pass fused=True as well")
    base = register(name)
    n = n_sig = 0
    for mod in model.modules():
        if hasattr(mod, "gpu_backend") and hasattr(mod, "cpu_backend"):
            sig = _cell_uses_siging(mod) if siging is None else bool(siging)
            mod.gpu_backend = mLSTMBackend(mLSTMBackendConfig(
                chunkwise_kernel=base + ("_siging" if sig else ""), sequence_kernel="native_sequence__native",
                step_kernel="native", mode=mode, return_last_states=False, chunk_size=64, eps=1e-6,
                autocast_kernel_dtype="bfloat16"))
            n += 1
            n_sig += int(sig)
    if keep_activations:
        for mod in model.modules():
            if hasattr(mod, "ckpt_thresh"):
                mod.ckpt_thresh = 1 << 62
    if fused:
        from . import vil

        vil.patch_layers(model, siging=siging, kernel_dtype=kernel_dtype, graphs=graphs)
    return n


from . import ops as _ops  # noqa: E402  (the torch.library ops are built on this module's launchers)
