"""The sigmoid-input-gate mLSTM without its normaliser (``normalize=False``) without a device: the chunkwise float64
reference of the tests (``tests/unnormalized_oracle.py``, on the oracle's primitives) against two independent float64
formulations (the parallel quadratic form and a token-by-token recurrence), its backward against autograd of the
quadratic form (without a normaliser and a max state the custbw-style backward is the exact derivative), and the
argument plumbing of the public entry points and the torch.library fakes."""
import os
import sys

import pytest
import torch
import torch.nn.functional as F

from oracle import mlstm_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import unnormalized_oracle as U  # noqa: E402

SEQ_LENS = [4, 16, 64]


def _inputs(S, DK, DV, seed, states):
    inp = O.make_inputs(2, 3, S, DK, DV, seed=seed, dtype=torch.float64, with_states=states)
    inp.pop("m0", None)  # the sigmoid-input-gate cell has no max state
    return inp


def quadratic(q, k, v, i, f, c0=None, n0=None):
    """h = ((Q K^T scale) . D) V + exp(F_t) scale q_t^T C0 with D_ts = exp(F_t - F_s + logsigmoid(i_s)) (s <= t),
    F_t = sum_{r <= t} logsigmoid(f_r), over the whole sequence at once; plus the last states (C, n)."""
    B, NH, S, DK = q.shape
    scale = DK ** -0.5
    Fc = torch.cumsum(F.logsigmoid(f), -1)
    li = F.logsigmoid(i)
    logd = Fc[..., :, None] - Fc[..., None, :] + li[..., None, :]
    causal = torch.ones(S, S, dtype=torch.bool).tril()
    D = torch.exp(logd.masked_fill(~causal, float("-inf")))
    h = ((q @ k.transpose(-1, -2)) * scale * D) @ v
    w_last = torch.exp(Fc[..., -1:] - Fc + li)  # weight of token s in the last state
    C = torch.einsum("bhs,bhsd,bhse->bhde", w_last, k, v)
    n = torch.einsum("bhs,bhsd->bhd", w_last, k)
    if c0 is not None:
        h = h + torch.exp(Fc)[..., None] * scale * (q @ c0)
        C = C + torch.exp(Fc[..., -1])[..., None, None] * c0
        n = n + torch.exp(Fc[..., -1])[..., None] * n0
    return h, C, n


def recurrence(q, k, v, i, f, c0=None, n0=None):
    """C_t = sigmoid(f_t) C_{t-1} + sigmoid(i_t) k_t v_t^T, n_t likewise, h_t = scale q_t^T C_t, token by token."""
    B, NH, S, DK = q.shape
    C = torch.zeros(B, NH, DK, v.shape[-1], dtype=q.dtype) if c0 is None else c0.clone()
    n = torch.zeros(B, NH, DK, dtype=q.dtype) if n0 is None else n0.clone()
    fg, ig = torch.sigmoid(f), torch.sigmoid(i)
    hs = []
    for t in range(S):
        C = fg[:, :, t, None, None] * C + ig[:, :, t, None, None] * (k[:, :, t, :, None] * v[:, :, t, None, :])
        n = fg[:, :, t, None] * n + ig[:, :, t, None] * k[:, :, t]
        hs.append(torch.einsum("bhd,bhde->bhe", q[:, :, t] * DK ** -0.5, C))
    return torch.stack(hs, 2), C, n


def _close(a, b, tol, what):
    e = O.rel_err(a, b)
    assert e < tol, f"{what}: rel err {e:.3e} >= {tol}"


@pytest.mark.parametrize("states", [False, True], ids=["plain", "states"])
@pytest.mark.parametrize("L", SEQ_LENS)
def test_reference_forward_matches_quadratic_form_and_recurrence(L, states):
    S = max(2 * L, 32)
    t = _inputs(S, 16, 24, seed=L + 100 * states, states=states)
    st = (t["c0"], t["n0"]) if states else (None, None)
    h, n_out, m_out, (C, n, m) = U.chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], *st, chunk_size=L)
    for name, ref in (("quadratic", quadratic), ("recurrence", recurrence)):
        h_r, C_r, n_r = ref(t["q"], t["k"], t["v"], t["i"], t["f"], *st)
        _close(h, h_r, 1e-12, f"h vs {name}")
        _close(C, C_r, 1e-12, f"C_last vs {name}")
        _close(n, n_r, 1e-12, f"n_last vs {name}")
    assert torch.all(m_out == 0) and torch.all(m == 0)
    # n_out and the states are those of the normalised call; only h differs, by the normaliser
    h1, n1, m1, (C1, nl1, _), _ = O.chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], *st, None, chunk_size=L,
                                                 siging=True)
    assert torch.equal(n_out, n1) and torch.equal(m_out, m1) and torch.equal(C, C1) and torch.equal(n, nl1)
    _close(h1, h / (n_out[..., None] + 1e-6), 1e-14, "normalised h = h / (n_out + eps)")


@pytest.mark.parametrize("states", [False, True], ids=["plain", "states"])
@pytest.mark.parametrize("L", SEQ_LENS)
def test_reference_backward_is_the_exact_derivative(L, states):
    """dq, dk, dv, di, df (and dC_initial) of the chunkwise backward against torch.autograd.grad of the quadratic form.
    With initial states the loss also has a C_last term, except for df: the chunkwise backward's dF (a reverse cumulative
    sum of q.dq - k.dk, bw.py:319-327) leaves out the C_last gradient of the forget gates in every variant, so df is
    compared without it."""
    S = max(2 * L, 32)
    t = _inputs(S, 16, 24, seed=7 * L + states, states=states)
    x = {n: t[n].clone().requires_grad_(True) for n in ("q", "k", "v", "i", "f")}
    st = (t["c0"].clone().requires_grad_(True), t["n0"]) if states else (None, None)
    dcl = t["dc_last"] if states else None

    def loss(with_c_last):
        h, C, _ = quadratic(x["q"], x["k"], x["v"], x["i"], x["f"], *st)
        out = (h * t["dh"]).sum()
        return out + (C * dcl).sum() if (with_c_last and dcl is not None) else out

    wrt = [x[n] for n in ("q", "k", "v", "i")] + ([st[0]] if states else [])
    g_ref = torch.autograd.grad(loss(True), wrt)
    (df_ref,) = torch.autograd.grad(loss(False), [x["f"]])
    g = U.chunkwise_bw(t["q"], t["k"], t["v"], t["i"], t["f"], t["dh"], *st, dcl, chunk_size=L)
    names = ["dq", "dk", "dv", "di"] + (["dc0"] if states else [])
    got = list(g[:4]) + ([g[5]] if states else [])
    for name, a, b in zip(names, got, g_ref):
        _close(a, b, 1e-10, name)
    if states:
        g = U.chunkwise_bw(t["q"], t["k"], t["v"], t["i"], t["f"], t["dh"], *st, None, chunk_size=L)
    _close(g[4], df_ref, 1e-10, "df")


# ---------------------------------------------------------------------------------------------------------------------
# public entry points without a device
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as G

    G.build()
    import xlstm_yolo_clean_b200 as p

    return p


def _cpu(S=64, DK=32, DV=32, dtype=torch.bfloat16):
    t = O.make_inputs(1, 2, S, DK, DV, seed=0, dtype=dtype)
    return t["q"], t["k"], t["v"], t["i"], t["f"]


def test_dropin_normalize_false_reaches_the_device_check(pkg):
    q, k, v, i, f = _cpu()
    with pytest.raises(RuntimeError, match="no CPU path"):
        pkg.mlstm_siging_chunkwise__b200(q, k, v, i, f, normalize=False)
    with pytest.raises(RuntimeError, match="no CPU path"):
        pkg.mlstm_siging_chunkwise__b200(q, k, v, i, f, normalize=False, return_last_states=True)


def test_exp_gate_without_normaliser_is_a_value_error(pkg):
    q, k, v, i, f = _cpu()
    with pytest.raises(ValueError, match="sigmoid input gate"):
        pkg.mlstm_chunkwise_fw(q, k, v, i, f, normalize=False)
    with pytest.raises(ValueError, match="sigmoid input gate"):
        pkg.mlstm_chunkwise_bw(q, k, v, i, f, q[..., 0].float(), q[..., 0].float(), v, normalize=False)
    with pytest.raises(ValueError, match="sigmoid input gate"):
        pkg.mlstm_recurrent_sequence__b200(q, k, v, i, f, normalize=False)
    for fn in (pkg.mlstm_chunkwise_fw, pkg.mlstm_recurrent_sequence__b200):  # the sigmoid-gate call gets to the device check
        with pytest.raises(RuntimeError, match="no CPU path"):
            fn(q, k, v, i, f, siging=True, normalize=False)


def test_cabi_refuses_bad_siging_and_unnormalised_epilogue(pkg):
    """The C-ABI checks the mode before it looks for a device: any value but 0 / 1 / 2 is EINVAL, and the fused
    cell-output epilogue with siging = 2 is EUNSUPPORTED.  (The pointers are never dereferenced.)"""
    import ctypes

    from xlstm_yolo_clean_b200 import _cabi

    lib = pkg.load_library()
    a = _cabi.FwArgs()
    s = a.shape
    s.B, s.NH, s.S, s.DHQK, s.DHHV, s.chunk_size, s.dtype = 1, 1, 64, 64, 64, 64, _cabi.BF16
    for name in ("q", "k", "v", "i", "f", "h"):
        t = getattr(a, name)
        t.ptr = 4096
        t.stride[:4] = (64 * 64, 64 * 64, 64, 1)
    a.n_out = a.m_out = 4096
    s.siging = 3
    assert lib.mlstm_b200_chunkwise_fw(ctypes.byref(a), None) == -1
    assert b"siging" in lib.mlstm_b200_last_error()
    e = _cabi.FwEpilogue()
    e.y.ptr = 4096
    e.y.stride[:4] = (64 * 64, 64 * 64, 64, 1)
    e.xy_dtype = _cabi.BF16
    a.epilogue = ctypes.pointer(e)
    s.siging = 2
    assert lib.mlstm_b200_chunkwise_fw(ctypes.byref(a), None) == -2
    assert b"epilogue" in lib.mlstm_b200_last_error()
    r = _cabi.RecurrentArgs()
    r.siging = -1
    assert lib.mlstm_b200_recurrent_sequence(ctypes.byref(r), None) == -1


def _sig(out):
    return [(tuple(t.shape), t.stride(), t.dtype, t.device.type) for t in out]


CASES = [(32, 32, torch.bfloat16), (64, 64, torch.bfloat16), (128, 128, torch.bfloat16), (32, 64, torch.bfloat16),
         (64, 128, torch.bfloat16), (64, 64, torch.float32)]  # the last: exact (FFMA) route


@pytest.mark.parametrize("DK,DV,dtype", CASES)
def test_op_fakes_allocate_the_same_with_normalize_false(pkg, DK, DV, dtype):
    from torch._subclasses.fake_tensor import FakeTensorMode

    ops = torch.ops.mlstm_b200
    B, NH, S = 3, 2, 320
    with FakeTensorMode():
        mk = lambda *s, dt=dtype: torch.empty(*s, device="cuda", dtype=dt)  # noqa: E731
        q, k, v, i, f = mk(B, NH, S, DK), mk(B, NH, S, DK), mk(B, NH, S, DV), mk(B, NH, S), mk(B, NH, S)
        c0, n0 = mk(B, NH, DK, DV, dt=torch.float32), mk(B, NH, DK, dt=torch.float32)
        for save, last in ((True, True), (False, False)):
            fw = (q, k, v, i, f, c0, n0, None, None, None, last, 64, 1e-6, 0, save, False, True, 0.0, None)
            base = _sig(ops.chunkwise_fw(*fw))
            assert _sig(ops.chunkwise_fw(*fw, True)) == base
            assert _sig(ops.chunkwise_fw(*fw, normalize=False)) == base
        nm = mk(2, B, NH, S, dt=torch.float32)
        bw = (q, k, v, i, f, nm[0], nm[1], v, c0, n0, None, None, None, None, None, 64, 1e-6, 0, True, False, True, 0.0,
              None)
        base = _sig(ops.chunkwise_bw(*bw))
        assert _sig(ops.chunkwise_bw(*bw, normalize=False)) == base
        rs = (q, k, v, i, f, c0, n0, None, True, 1e-6, True)
        base = _sig(ops.recurrent_sequence(*rs))
        assert _sig(ops.recurrent_sequence(*rs, normalize=False)) == base
        with pytest.raises(ValueError):  # the exp gate has no unnormalised form, in the fakes too
            ops.chunkwise_fw(*fw[:16], False, *fw[17:], normalize=False)
