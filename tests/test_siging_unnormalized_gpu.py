"""The sigmoid-input-gate mLSTM without its normaliser (``normalize=False``, C-ABI ``siging = 2``) on the B200: every
kernel family that implements the sigmoid input gate -- the tensor-core forward (tc_fw, tc_fw_d128, tc_fw_rect) and
backward (tc_bw, also as the block problems of head dim 128 and of rectangular heads), the exact fp32 kernels and the
recurrent kernels -- against the float64 oracle on inputs rounded to the test dtype (max|a-b| / max|b| per tensor:
2e-2 for 16-bit, 1e-5 for fp32), plus the public entry points, torch.compile and the refusals."""
import math
import os
import sys

import pytest
import torch

from oracle import mlstm_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import unnormalized_oracle as U  # noqa: E402

pytestmark = pytest.mark.gpu

PAIRS = [(32, 32), (64, 64), (128, 128), (32, 64), (64, 128)]
PAIR_IDS = ["d32", "d64", "d128", "qk32_v64", "qk64_v128"]
ROUTES = [(torch.bfloat16, 2e-2), (torch.float16, 2e-2), (torch.float32, 1e-5)]
ROUTE_IDS = ["bf16", "fp16", "fp32"]
SEQ = ("q", "k", "v", "i", "f", "dh")


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as G

    G.build()
    import xlstm_yolo_clean_b200 as p

    return p


def _inputs(B, NH, S, DK, DV, seed, states):
    """SURVEY.md section 8(d) inputs (q, k, v, i ~ N(0, 1), f ~ N(3, 1)): the forget window of ~20 tokens keeps the
    unnormalised h well inside the fp16 range.  No m_initial: the sigmoid-input-gate cell has no max state."""
    inp = O.make_inputs(B, NH, S, DK, DV, seed=seed, dtype=torch.float32, with_states=states)
    inp.pop("m0", None)
    return inp


def _dev(inp, dtype):
    return {k: v.to(dtype).cuda() for k, v in inp.items()}


def _fwbw(pkg, t, L, reverse=False, states=False, normalize=False, save_states=True, n_out_override=None):
    kw = dict(c_initial=t["c0"], n_initial=t["n0"]) if states else {}
    h, n_out, m_out, last, cst = pkg.mlstm_chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=L,
                                                        return_last_states=states, reverse=reverse, siging=True,
                                                        normalize=normalize, save_states=save_states, **kw)
    n_fw = pkg.last_launch_count()
    if n_out_override is not None:
        n_out = n_out_override
    g = pkg.mlstm_chunkwise_bw(t["q"], t["k"], t["v"], t["i"], t["f"], n_out, m_out, t["dh"], chunk_size=L, c_states=cst,
                               reverse=reverse, siging=True, normalize=normalize,
                               dc_last=t["dc_last"] if states else None, want_dc_initial=states, **kw)
    n_bw = pkg.last_launch_count()
    torch.cuda.synchronize()
    out = dict(h=h, dq=g[0], dk=g[1], dv=g[2], di=g[3], df=g[4])
    if states:
        out.update(c_last=last[0], n_last=last[1], dc0=g[5])
    return out, cst, (n_fw, n_bw)


def _oracle(inp, dtype, L, reverse=False, states=False):
    """The float64 unnormalised reference (tests/unnormalized_oracle.py) on the inputs rounded to ``dtype``."""
    r = {k: v.to(dtype).double() for k, v in inp.items()}
    if reverse:
        r = {k: (v.flip(2) if k in SEQ else v) for k, v in r.items()}
    st = (r["c0"], r["n0"]) if states else (None, None)
    h, last, g = U.fwbw(r["q"], r["k"], r["v"], r["i"], r["f"], r["dh"], *st, dc_last=r["dc_last"] if states else None,
                        chunk_size=L)
    out = dict(h=h, dq=g[0], dk=g[1], dv=g[2], di=g[3], df=g[4])
    if reverse:
        out = {k: v.flip(2) for k, v in out.items()}
    if states:
        out.update(c_last=last[0], n_last=last[1], dc0=g[5])
    return out


def _assert_close(got, want, tol, what):
    bad = {}
    for k, w in want.items():
        e = O.rel_err(got[k].double().cpu().reshape(w.shape), w)
        if not e < tol:
            bad[k] = e
    assert not bad, f"{what}: rel err above {tol}: {bad}"


def _route_shape(dtype):
    """16-bit: the tensor route at a ragged S (196 = one full and one 68-token tile, chunk 4); fp32: the exact route."""
    return (196, 4) if dtype != torch.float32 else (192, 64)


@pytest.mark.parametrize("states", [False, True], ids=["plain", "states"])
@pytest.mark.parametrize("reverse", [False, True], ids=["causal", "anticausal"])
@pytest.mark.parametrize("dtype,tol", ROUTES, ids=ROUTE_IDS)
@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_parity_with_oracle(pkg, DK, DV, dtype, tol, reverse, states):
    """h, dq, dk, dv, di, df -- with initial states and dC_last also C_last, n_last and dC_initial."""
    S, L = _route_shape(dtype)
    if dtype != torch.float32:
        assert pkg.tensor_path_supported(2, 2, S, DK, DV, dtype, chunk_size=L)
    inp = _inputs(2, 2, S, DK, DV, seed=DK + DV + 7 * reverse + 3 * states, states=states)
    got, cst, (n_fw, _) = _fwbw(pkg, _dev(inp, dtype), L, reverse, states)
    assert (cst is not None) == (dtype != torch.float32)  # the 16-bit calls ran on the tensor route
    _assert_close(got, _oracle(inp, dtype, L, reverse, states), tol, f"({DK}, {DV}) {dtype}")


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_backward_does_not_read_n_out(pkg, DK, DV, dtype):
    """The backward of the unnormalised call gives the same gradients, bit for bit, when n_out is all NaN."""
    S, L = _route_shape(dtype)
    inp = _inputs(2, 2, S, DK, DV, seed=40 + DK, states=True)
    t = _dev(inp, dtype)
    a, _, _ = _fwbw(pkg, t, L, states=True)
    nan = torch.full((2, 2, S), math.nan, device="cuda")
    b, _, _ = _fwbw(pkg, t, L, states=True, n_out_override=nan)
    for k in a:
        assert torch.equal(a[k], b[k]), k
    c, _, _ = _fwbw(pkg, t, L, states=True, save_states=False, n_out_override=nan)  # recomputed states
    for k in ("dq", "dk", "dv", "di", "df", "dc0"):
        assert torch.equal(a[k], c[k]), k


def _bshd(t, dt):
    """q / k as the two halves of one (B, S, NH, 2 DHQK) tensor and v / dh with their own (B, S, NH, DHHV) token stride,
    the views MatrixLSTMCell.forward hands over (vision_lstm2.py:718-727)."""
    B, NH, S, DK = t["q"].shape
    qk = torch.empty(B, S, NH, 2 * DK, dtype=dt, device="cuda")
    qk[..., :DK] = t["q"].transpose(1, 2)
    qk[..., DK:] = t["k"].transpose(1, 2)
    out = dict(t)
    out["q"], out["k"] = qk[..., :DK].transpose(1, 2), qk[..., DK:].transpose(1, 2)
    out["v"] = t["v"].transpose(1, 2).contiguous().transpose(1, 2)
    out["dh"] = t["dh"].transpose(1, 2).contiguous().transpose(1, 2)
    assert not out["q"].is_contiguous() and not out["v"].is_contiguous()
    return out


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("DK,DV", [(64, 64), (128, 128), (32, 64)], ids=["d64", "d128", "qk32_v64"])
def test_strided_bshd_views_ragged_sequence(pkg, DK, DV, dtype):
    """Strided views at a ragged S = 324 (two full tiles and a 68-token one) with chunk size 4, taken as they are."""
    S, L = 324, 4
    inp = _inputs(2, 3, S, DK, DV, seed=90 + DK, states=True)
    t = _bshd(_dev(inp, dtype), dtype)
    got, cst, _ = _fwbw(pkg, t, L, states=True)
    assert cst is not None
    _assert_close(got, _oracle(inp, dtype, L, states=True), 2e-2, f"strided ({DK}, {DV}) {dtype}")


@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_tensor_route_agrees_with_exact_route(pkg, DK, DV):
    """The same bf16 call through the exact fp32 FFMA kernels and through the tensor route."""
    inp = _inputs(2, 3, 384, DK, DV, seed=11 + DK, states=True)
    t = _dev(inp, torch.bfloat16)
    pkg.set_default_impl("exact")
    try:
        ex, cst_ex, _ = _fwbw(pkg, t, 64, states=True)
    finally:
        pkg.set_default_impl("auto")
    tc, cst_tc, _ = _fwbw(pkg, t, 64, states=True)
    assert cst_ex is None and cst_tc is not None  # EXACT took the FFMA kernels, AUTO the tensor route
    for k in tc:
        assert O.rel_err(tc[k].double().cpu(), ex[k].double().cpu()) < 2e-2, k


def test_fp16_autocast_bf16_kernel_writes_fp16_gradients(pkg):
    """The drop-in under fp16 autocast with the default bf16 kernel: custom_fwd rounds the inputs to bf16, the backward
    writes the fp16 gradients straight from the kernel (grad_dtype)."""
    B, NH, S, D = 2, 3, 324, 64
    inp = _inputs(B, NH, S, D, D, seed=21, states=False)
    leaves = {k: inp[k].to(torch.float16).cuda().requires_grad_(True) for k in ("q", "k", "v", "i", "f")}
    dh = inp["dh"].to(torch.float16).to(torch.bfloat16).cuda()
    with torch.autocast("cuda", dtype=torch.float16):
        h = pkg.mlstm_siging_chunkwise__b200(**leaves, chunk_size=4, normalize=False)
    assert h.dtype == torch.bfloat16
    h.backward(dh)
    torch.cuda.synchronize()
    rounded = {k: v.to(torch.float16).to(torch.bfloat16) for k, v in inp.items()}
    want = _oracle(rounded, torch.bfloat16, 4)
    got = dict(h=h, **{"d" + k: leaves[k].grad for k in leaves})
    assert all(leaves[k].grad.dtype == torch.float16 for k in leaves)
    _assert_close(got, want, 2e-2, "fp16 autocast")


@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_launch_counts_and_repeatability(pkg, DK, DV):
    """The unnormalised call launches exactly what the normalised one does -- forward, backward with the saved states,
    backward that recomputes them (the head-dim-128 and rectangular block problems included) -- and two identical calls
    agree bit for bit."""
    inp = _inputs(2, 2, 324, DK, DV, seed=5, states=True)
    t = _dev(inp, torch.bfloat16)
    counts = {}
    runs = {}
    for normalize in (True, False):
        for save in (True, False):
            a, _, na = _fwbw(pkg, t, 4, states=True, normalize=normalize, save_states=save)
            b, _, nb = _fwbw(pkg, t, 4, states=True, normalize=normalize, save_states=save)
            assert na == nb
            for k in a:
                assert torch.equal(a[k], b[k]), (normalize, save, k)
            counts[normalize, save] = na
            runs[normalize, save] = a
    assert counts[False, True] == counts[True, True]
    assert counts[False, False] == counts[True, False]
    for k in runs[False, True]:  # saved and recomputed states give the same unnormalised gradients
        assert torch.equal(runs[False, True][k], runs[False, False][k]), k
    assert not torch.equal(runs[False, True]["h"], runs[True, True]["h"])


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_explicit_normalize_true_is_the_default(pkg, dtype):
    inp = _inputs(2, 3, 256, 64, 64, seed=8, states=True)

    def run(**kw):
        x = {k: inp[k].to(dtype).cuda().requires_grad_(True) for k in ("q", "k", "v", "i", "f")}
        c0 = inp["c0"].cuda().requires_grad_(True)
        h, (c, n) = pkg.mlstm_siging_chunkwise__b200(**x, c_initial=c0, n_initial=inp["n0"].cuda(),
                                                     return_last_states=True, **kw)
        torch.autograd.backward([h, c], [inp["dh"].to(dtype).cuda(), inp["dc_last"].to(dtype).cuda()])
        torch.cuda.synchronize()
        return [h, c, n] + [x[k].grad for k in x] + [c0.grad]

    for a, b in zip(run(), run(normalize=True)):
        assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------------ recurrent kernels
def _recurrence(r):
    """Float64 token-by-token cell without the normaliser: h_t = DHQK^-1/2 q_t^T C_t."""
    q, k, v, i, f = r["q"], r["k"], r["v"], r["i"], r["f"]
    C, n = r["c0"].clone(), r["n0"].clone()
    fg, ig = torch.sigmoid(f), torch.sigmoid(i)
    hs = []
    for t in range(q.shape[2]):
        C = fg[:, :, t, None, None] * C + ig[:, :, t, None, None] * (k[:, :, t, :, None] * v[:, :, t, None, :])
        n = fg[:, :, t, None] * n + ig[:, :, t, None] * k[:, :, t]
        hs.append(torch.einsum("bhd,bhde->bhe", q[:, :, t] * q.shape[-1] ** -0.5, C))
    return torch.stack(hs, 2), C, n


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-5), (torch.bfloat16, 2e-2)], ids=["fp32", "bf16"])
@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_recurrent_sequence_matches_recurrence(pkg, DK, DV, dtype, tol):
    inp = _inputs(2, 3, 40, DK, DV, seed=11 + DK, states=True)
    h_ref, c_ref, n_ref = _recurrence({k: v.to(dtype).double() for k, v in inp.items()})
    t = _dev(inp, dtype)
    h, (c, n, m) = pkg.mlstm_recurrent_sequence__b200(t["q"], t["k"], t["v"], t["i"], t["f"], inp["c0"].cuda(),
                                                      inp["n0"].cuda(), None, return_last_states=True, siging=True,
                                                      normalize=False)
    torch.cuda.synchronize()
    assert torch.all(m == 0)
    for name, a, b in (("h", h, h_ref), ("c", c, c_ref), ("n", n, n_ref)):
        assert O.rel_err(a.double().cpu(), b) < tol, name


def test_step_kernel_chains_like_the_sequence(pkg):
    B, NH, S, DK, DV = 2, 4, 9, 64, 128
    inp = _inputs(B, NH, S, DK, DV, seed=3, states=True)
    t = _dev(inp, torch.float32)
    kw = dict(siging=True, normalize=False)
    h_seq, (c_seq, n_seq, _) = pkg.mlstm_recurrent_sequence__b200(t["q"], t["k"], t["v"], t["i"], t["f"], t["c0"], t["n0"],
                                                                  None, return_last_states=True, **kw)
    c, n, m = t["c0"], t["n0"], torch.zeros(B, NH, 1, device="cuda")
    hs = []
    for s in range(S):
        h, (c, n, m) = pkg.mlstm_recurrent_step__b200(t["q"][:, :, s], t["k"][:, :, s], t["v"][:, :, s],
                                                       t["i"][:, :, s, None], t["f"][:, :, s, None], c, n, m, **kw)
        hs.append(h)
    torch.cuda.synchronize()
    assert torch.equal(torch.stack(hs, 2), h_seq) and torch.equal(c, c_seq) and torch.equal(n, n_seq)


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-5), (torch.bfloat16, 2e-2)], ids=["fp32", "bf16"])
@pytest.mark.parametrize("DK,DV", [(64, 64), (32, 64)], ids=["d64", "qk32_v64"])
def test_chunkwise_prefix_continues_in_the_recurrent_kernel(pkg, DK, DV, dtype, tol):
    """A return_last_states prefix of the drop-in, continued token by token by the recurrent sequence kernel with the
    same function, equals the chunkwise call over the whole sequence."""
    S0, S1 = 128, 64
    inp = _inputs(2, 3, S0 + S1, DK, DV, seed=31, states=False)
    t = _dev(inp, dtype)
    full = pkg.mlstm_siging_chunkwise__b200(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=64, normalize=False)
    pre = {k: t[k][:, :, :S0] for k in ("q", "k", "v", "i", "f")}
    rest = {k: t[k][:, :, S0:] for k in ("q", "k", "v", "i", "f")}
    h0, (c, n) = pkg.mlstm_siging_chunkwise__b200(**pre, chunk_size=64, normalize=False, return_last_states=True)
    h1 = pkg.mlstm_recurrent_sequence__b200(**rest, c_initial=c, n_initial=n, siging=True, normalize=False)
    torch.cuda.synchronize()
    assert O.rel_err(torch.cat([h0, h1], 2).double().cpu(), full.double().cpu()) < tol
    assert O.rel_err(h1.double().cpu(), full[:, :, S0:].double().cpu()) < tol


# ------------------------------------------------------------------------------------------------ refusals, compile
def test_fused_epilogue_is_refused(pkg):
    from xlstm_yolo_clean_b200 import backend

    B, NH, S, D = 1, 2, 128, 64
    inp = _dev(_inputs(B, NH, S, D, D, seed=1, states=False), torch.bfloat16)
    y = torch.empty(B, NH, S, D, device="cuda", dtype=torch.bfloat16)
    epi = backend.FwEpilogue(y, None, None, None, None, 1e-5, False)
    args = (inp["q"], inp["k"], inp["v"], inp["i"], inp["f"], None, None, None, None, False, 64, 1e-6, None, False, False)
    backend._fw_launch(*args, 1, 0.0, epi)  # the normalised sigmoid-gate cell is covered
    with pytest.raises(RuntimeError, match="siging = 2"):
        backend._fw_launch(*args, 2, 0.0, epi)


def test_opcheck_unnormalised_ops(pkg):
    ops = torch.ops.mlstm_b200
    inp = _dev(_inputs(2, 2, 128, 64, 64, seed=2, states=False), torch.bfloat16)
    q, k, v, i, f = (inp[n].requires_grad_(True) for n in ("q", "k", "v", "i", "f"))
    fw = (q, k, v, i, f, None, None, None, None, None, True, 64, 1e-6, 0, True, False, True, 0.0, None, False)
    torch.library.opcheck(ops.chunkwise_fw, fw)
    h, nm, _, _, _, cs = (x.detach() for x in ops.chunkwise_fw(*fw))
    qd, kd, vd, idd, fd = (x.detach() for x in (q, k, v, i, f))
    torch.library.opcheck(ops.chunkwise_bw, (qd, kd, vd, idd, fd, nm[0], nm[1], torch.randn_like(h), None, None, None, None,
                                             cs, None, None, 64, 1e-6, 0, False, False, True, 0.0, None, False))
    torch.library.opcheck(ops.recurrent_sequence, (qd[:, :, :16], kd[:, :, :16], vd[:, :, :16], idd[:, :, :16],
                                                   fd[:, :, :16], None, None, None, True, 1e-6, True, False))


@pytest.mark.parametrize("states", [False, True], ids=["plain", "states"])
@pytest.mark.parametrize("DK,DV", [(64, 64), (128, 128), (32, 64)], ids=["d64", "d128", "qk32_v64"])
def test_compile_fullgraph_matches_eager(pkg, DK, DV, states):
    torch._dynamo.reset()
    B, NH, S = 2, 3, 192
    inp = _inputs(B, NH, S, DK, DV, seed=DK + states, states=states)

    def fn(q, k, v, i, f, *st):
        kw = dict(zip(("c_initial", "n_initial"), st))
        out = pkg.mlstm_siging_chunkwise__b200(q, k, v, i, f, chunk_size=64, normalize=False,
                                               return_last_states=states, **kw)
        return (out[0], *out[1]) if states else (out,)

    def run(f_):
        ts = [inp[n].to(torch.bfloat16).cuda().requires_grad_(True) for n in ("q", "k", "v", "i", "f")]
        if states:
            ts += [inp["c0"].cuda().requires_grad_(True), inp["n0"].cuda()]
        outs = f_(*ts)
        douts = [inp["dh"].to(torch.bfloat16).cuda()] + ([inp["dc_last"].to(torch.bfloat16).cuda()] if states else [])
        torch.autograd.backward(list(outs[:len(douts)]), douts)
        torch.cuda.synchronize()
        return [o.detach() for o in outs] + [t.grad for t in ts if t.requires_grad]

    ts = [inp[n].to(torch.bfloat16).cuda() for n in ("q", "k", "v", "i", "f")]
    ex = torch._dynamo.explain(fn)(*ts, *([inp["c0"].cuda(), inp["n0"].cuda()] if states else []))
    assert ex.graph_break_count == 0 and ex.graph_count == 1, ex.break_reasons
    torch._dynamo.reset()
    eager = run(fn)
    compiled = run(torch.compile(fn, fullgraph=True))
    try:
        for a, b in zip(eager, compiled):
            assert a.dtype == b.dtype and torch.equal(a, b)
    finally:
        torch._dynamo.reset()
