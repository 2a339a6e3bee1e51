"""Head dims above 128 on the exact (fp32 FFMA) route: every DHQK <= 256, DHHV <= 512 (multiples of 4), with xLSTM-Large's
(256, 512) in fp32 -- the model run without autocast -- as the main case.  k_fw_h writes h in column blocks of v and
k_bw_dqkv sums dS, dI and the inter-chunk parts of dQ / dK over them in shared memory, so the launch counts (forward 2,
backward 4) and the fixed summation order (bit-identical repeats) are those of the narrower heads.  Everything is
measured against the float64 oracle on inputs rounded to the test dtype (max|a-b| / max|b| per tensor: 1e-5 in fp32,
2e-2 in 16-bit); B * NH <= 2 and S <= 512 keep the oracle cheap, except in the one large-index test."""
import ctypes
import os
import sys

import pytest
import torch

from oracle import mlstm_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import unnormalized_oracle as U  # noqa: E402

pytestmark = pytest.mark.gpu
PAIRS = [(256, 512), (256, 256), (128, 256), (128, 512), (132, 260)]
PAIR_IDS = [f"{dk}x{dv}" for dk, dv in PAIRS]
SEQ = ("q", "k", "v", "i", "f", "dh")
MODES = [0, 1, 2]  # C-ABI siging: exponential input gate, sigmoid input gate, sigmoid input gate without normaliser
MODE_IDS = ["exp", "siging", "siging_unnorm"]
F32_TOL, HALF_TOL = 1e-5, 2e-2


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as G

    G.build()
    import xlstm_yolo_clean_b200 as p

    return p


def _inputs(B, NH, S, DK, DV, seed, states, mode=0):
    inp = O.make_inputs(B, NH, S, DK, DV, seed=seed, dtype=torch.float32, with_states=states)
    if states and mode:  # the sigmoid-input-gate cell has no max state
        inp["m0"] = torch.zeros_like(inp["m0"])
    return inp


def _api(mode):
    return dict(siging=mode != 0, normalize=mode != 2)


def _fwbw(pkg, t, L, reverse=False, mode=0, states=False):
    kw = dict(c_initial=t["c0"], n_initial=t["n0"], m_initial=t["m0"]) if states else {}
    h, n_out, m_out, last, cst = pkg.mlstm_chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=L,
                                                        return_last_states=states, reverse=reverse, **_api(mode), **kw)
    n_fw = pkg.last_launch_count()
    g = pkg.mlstm_chunkwise_bw(t["q"], t["k"], t["v"], t["i"], t["f"], n_out, m_out, t["dh"], chunk_size=L, c_states=cst,
                               reverse=reverse, dc_last=t["dc_last"] if states else None, want_dc_initial=states,
                               **_api(mode), **kw)
    n_bw = pkg.last_launch_count()
    torch.cuda.synchronize()
    out = dict(h=h, dq=g[0], dk=g[1], dv=g[2], di=g[3], df=g[4])
    if states:
        out.update(c_last=last[0], n_last=last[1], m_last=last[2], dc0=g[5])
    return out, cst, (n_fw, n_bw)


def _oracle(inp, dtype, L, reverse=False, mode=0, states=False):
    r = {k: v.to(dtype).double() for k, v in inp.items()}
    if reverse:
        r = {k: (v.flip(2) if k in SEQ else v) for k, v in r.items()}
    dcl = r["dc_last"] if states else None
    if mode == 2:
        c0, n0 = (r["c0"], r["n0"]) if states else (None, None)
        h, last, g = U.fwbw(r["q"], r["k"], r["v"], r["i"], r["f"], r["dh"], c0, n0, dc_last=dcl, chunk_size=L)
    else:
        st = (r["c0"], r["n0"], r["m0"]) if states else (None, None, None)
        h, last, g = O.fwbw(r["q"], r["k"], r["v"], r["i"], r["f"], r["dh"], *st, dc_last=dcl, chunk_size=L, siging=mode == 1)
    out = dict(h=h, dq=g[0], dk=g[1], dv=g[2], di=g[3], df=g[4])
    if reverse:
        out = {k: v.flip(2) for k, v in out.items()}
    if states:
        out.update(c_last=last[0], n_last=last[1], m_last=last[2].reshape(-1), dc0=g[5])
    return out


def _assert_close(got, want, tol, what):
    bad = {}
    for k, w in want.items():
        e = O.rel_err(got[k].double().cpu().reshape(w.shape), w)
        if not e < tol:
            bad[k] = e
    assert not bad, f"{what}: rel err above {tol}: {bad}"


@pytest.mark.parametrize("L,S", [(64, 256), (16, 128)], ids=["chunk64", "chunk16"])
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("reverse", [False, True], ids=["causal", "anticausal"])
@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_fp32_parity_with_states(pkg, DK, DV, reverse, mode, L, S):
    """h, dq, dk, dv, di, df, the last states and dC_initial -- with initial states and dC_last -- over S / L = 4 and 8
    chunks."""
    inp = _inputs(1, 2, S, DK, DV, seed=DK + DV + 7 * reverse + 3 * mode + L, states=True, mode=mode)
    t = {k: v.cuda() for k, v in inp.items()}
    got, cst, launches = _fwbw(pkg, t, L, reverse, mode, states=True)
    assert cst is None and launches == (2, 4)
    _assert_close(got, _oracle(inp, torch.float32, L, reverse, mode, states=True), F32_TOL,
                  f"fp32 ({DK}, {DV}) chunk={L} reverse={reverse} siging={mode}")


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("DK,DV", PAIRS[1:], ids=PAIR_IDS[1:])
def test_16bit_pairs_off_the_tensor_route(pkg, DK, DV, dtype):
    """AUTO sends the 16-bit pairs the tensor-core route does not cover to the exact kernels."""
    S, L = 256, 64
    assert not pkg.tensor_path_supported(1, 2, S, DK, DV, dtype, chunk_size=L)
    inp = _inputs(1, 2, S, DK, DV, seed=DK * DV, states=True)
    t = {k: v.to(dtype).cuda() for k, v in inp.items()}
    got, cst, launches = _fwbw(pkg, t, L, states=True)
    assert cst is None and launches == (2, 4)
    _assert_close(got, _oracle(inp, dtype, L, states=True), HALF_TOL, f"{dtype} ({DK}, {DV})")


@pytest.mark.parametrize("reverse", [False, True], ids=["causal", "anticausal"])
def test_bf16_wide_pair_on_the_exact_route_by_choice(pkg, reverse):
    """set_default_impl("exact") takes bf16 (256, 512) off the tensor cores."""
    DK, DV, S, L = 256, 512, 256, 64
    inp = _inputs(1, 2, S, DK, DV, seed=99 + reverse, states=False)
    t = {k: v.to(torch.bfloat16).cuda() for k, v in inp.items()}
    pkg.set_default_impl("exact")
    try:
        got, cst, launches = _fwbw(pkg, t, L, reverse)
    finally:
        pkg.set_default_impl("auto")
    assert cst is None and launches == (2, 4)
    _assert_close(got, _oracle(inp, torch.bfloat16, L, reverse), HALF_TOL, "bf16 (256, 512) exact")


def test_fp32_dropin_autograd_with_last_states(pkg):
    """mlstm_chunkwise__b200 at fp32 (256, 512), return_last_states=True, backward through h and C_last."""
    DK, DV, S = 256, 512, 256
    inp = _inputs(1, 2, S, DK, DV, seed=21, states=True)
    ts = [inp[n].cuda().requires_grad_(True) for n in ("q", "k", "v", "i", "f")]
    h, (c, n, m) = pkg.mlstm_chunkwise__b200(*ts, chunk_size=64, return_last_states=True)
    assert h.dtype == torch.float32 and c.shape == (1, 2, DK, DV)
    torch.autograd.backward([h, c], [inp["dh"].cuda(), inp["dc_last"].cuda()])
    torch.cuda.synchronize()
    r = {k: v.double() for k, v in inp.items()}
    h_ref, last, g = O.fwbw(r["q"], r["k"], r["v"], r["i"], r["f"], r["dh"], dc_last=r["dc_last"], chunk_size=64)
    assert O.rel_err(h, h_ref) < F32_TOL
    for a, b, name in ((c, last[0], "c"), (n, last[1], "n"), (m.reshape(-1), last[2].reshape(-1), "m")):
        assert O.rel_err(a, b) < F32_TOL, name
    for x, w, name in zip(ts, g, ("dq", "dk", "dv", "di", "df")):
        assert x.grad.dtype == torch.float32 and O.rel_err(x.grad, w) < F32_TOL, name


def test_dropin_under_fp16_autocast_square_256(pkg):
    """(256, 256) under fp16 autocast: the bf16 kernel dtype on the exact route, fp16 gradients cast by autograd."""
    DK = DV = 256
    inp = _inputs(1, 2, 256, DK, DV, seed=13, states=False)
    ts = [inp[n].to(torch.float16).cuda().requires_grad_(True) for n in ("q", "k", "v", "i", "f")]
    with torch.autocast("cuda", dtype=torch.float16):
        h = pkg.mlstm_chunkwise__b200(*ts, chunk_size=64)
    assert pkg.last_launch_count() == 2
    h.backward(inp["dh"].to(torch.bfloat16).cuda())
    torch.cuda.synchronize()
    assert h.dtype == torch.bfloat16 and all(x.grad.dtype == torch.float16 for x in ts)
    r = {k: v.to(torch.float16).to(torch.bfloat16).double() for k, v in inp.items()}
    h_ref, _, g = O.fwbw(r["q"], r["k"], r["v"], r["i"], r["f"], r["dh"], chunk_size=64)
    assert O.rel_err(h, h_ref) < HALF_TOL
    for x, w, name in zip(ts, g, ("dq", "dk", "dv", "di", "df")):
        assert O.rel_err(x.grad, w) < HALF_TOL, name


def test_fp32_strided_and_offset_views(pkg):
    """xLSTM-Large's layout -- (B, S, NH, D) projections seen as (B, NH, S, D) -- and a view at an odd element offset
    of its storage, both taken as they are by the exact kernels."""
    DK, DV, S = 256, 512, 256
    inp = _inputs(1, 2, S, DK, DV, seed=90, states=False)
    t = {}
    for name, x in inp.items():
        if name in ("q", "k", "v", "dh"):
            B, NH, S_, D = x.shape
            x = x.cuda().transpose(1, 2).contiguous().view(B, S_, NH, D).transpose(1, 2)
            assert not x.is_contiguous()
        else:
            x = x.cuda()
        t[name] = x
    store = torch.empty(inp["v"].numel() + 1, device="cuda")
    t["v"] = store[1:].view(inp["v"].shape)
    t["v"].copy_(inp["v"])
    assert t["v"].data_ptr() % 16 == 4
    got, _, launches = _fwbw(pkg, t, 64)
    assert launches == (2, 4)
    _assert_close(got, _oracle(inp, torch.float32, 64), F32_TOL, "strided fp32 (256, 512)")


def test_bf16_offset_view_at_the_wide_pair_goes_exact(pkg):
    """A 16-bit (256, 512) view a TMA map cannot describe: the C-ABI sends it to the exact route under AUTO."""
    DK, DV, S = 256, 512, 128
    inp = _inputs(1, 2, S, DK, DV, seed=5, states=False)
    dt = torch.bfloat16
    lib, C = pkg.load_library(), pkg._cabi
    x = {k: inp[k].to(dt).cuda() for k in ("q", "k", "v", "i", "f")}
    st = torch.empty(inp["q"].numel() + 1, device="cuda", dtype=dt)
    q = st[1:].view(inp["q"].shape)
    q.copy_(x["q"])
    h = torch.empty(1, 2, S, DV, device="cuda", dtype=dt)
    nm = torch.empty(2, 1, 2, S, device="cuda")
    a = C.FwArgs()
    a.shape.B, a.shape.NH, a.shape.S, a.shape.DHQK, a.shape.DHHV = 1, 2, S, DK, DV
    a.shape.chunk_size, a.shape.dtype, a.shape.eps, a.shape.impl = 64, C.BF16, 1e-6, C.IMPL_AUTO
    for name, tt in (("q", q), ("k", x["k"]), ("v", x["v"]), ("i", x["i"]), ("f", x["f"]), ("h", h)):
        getattr(a, name).ptr = tt.data_ptr()
        getattr(a, name).stride[:tt.dim()] = tt.stride()
    a.n_out, a.m_out = nm[0].data_ptr(), nm[1].data_ptr()
    es = C.Shape()
    ctypes.memmove(ctypes.byref(es), ctypes.byref(a.shape), ctypes.sizeof(C.Shape))
    es.impl = C.IMPL_EXACT
    ws = torch.empty(lib.mlstm_b200_workspace_bytes(ctypes.byref(es), 0), device="cuda", dtype=torch.uint8)
    a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
    rc = lib.mlstm_b200_chunkwise_fw(ctypes.byref(a), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, lib.mlstm_b200_last_error()
    assert lib.mlstm_b200_last_launch_count() == 2
    torch.cuda.synchronize()
    r = {k: v.to(dt).double() for k, v in inp.items()}
    h_ref = O.chunkwise_fw(r["q"], r["k"], r["v"], r["i"], r["f"], chunk_size=64)[0]
    assert O.rel_err(h, h_ref) < HALF_TOL


def test_fp32_prefix_continued_by_the_sequence_kernel(pkg):
    """fp32 xLSTM-Large inference end to end: a chunkwise prefill with last states, continued token by token by
    mlstm_recurrent_sequence__b200, matches the oracle's step recurrence over the whole sequence."""
    DK, DV, S0, S1 = 256, 512, 256, 24
    inp = _inputs(1, 2, S0 + S1, DK, DV, seed=17, states=False)
    t = {k: v.cuda() for k, v in inp.items()}
    pre = {k: t[k][:, :, :S0] for k in ("q", "k", "v", "i", "f")}
    post = {k: t[k][:, :, S0:] for k in ("q", "k", "v", "i", "f")}
    h0, (c, n, m) = pkg.mlstm_chunkwise__b200(pre["q"], pre["k"], pre["v"], pre["i"], pre["f"], chunk_size=64,
                                              return_last_states=True)
    h1, (c1, n1, m1) = pkg.mlstm_recurrent_sequence__b200(post["q"], post["k"], post["v"], post["i"], post["f"], c, n, m,
                                                          return_last_states=True)
    torch.cuda.synchronize()
    r = {k: v.double() for k, v in inp.items()}
    h_ref, (c_ref, n_ref, m_ref) = O.step_recurrence(r["q"], r["k"], r["v"], r["i"], r["f"])
    assert O.rel_err(torch.cat([h0, h1], 2), h_ref) < F32_TOL
    for a, b, name in ((c1, c_ref, "c"), (n1, n_ref, "n"), (m1.reshape(-1), m_ref.reshape(-1), "m")):
        assert O.rel_err(a, b) < F32_TOL, name


def test_repeatable_and_launch_counts(pkg):
    """Two identical calls are bit-identical: the v blocks are summed in a fixed order, with no atomics."""
    DK, DV, S = 256, 512, 320
    inp = _inputs(1, 2, S, DK, DV, seed=8, states=True)
    t = {k: v.cuda() for k, v in inp.items()}
    a, _, la = _fwbw(pkg, t, 64, states=True)
    b, _, lb = _fwbw(pkg, t, 64, states=True)
    assert la == lb == (2, 4)
    for name in a:
        assert torch.equal(a[name], b[name]), name


def test_large_state_index(pkg):
    """fp32 (256, 512) at B * NH = 128, S = 4096: the internal chunk is 32 tokens, so the per-chunk state buffers hold
    128 * 129 * 256 * 512 > 2^31 elements.  The first and the last head get the same inputs and must give bit-identical
    outputs, which match the oracle."""
    DK, DV, NH, S, L = 256, 512, 128, 4096, 64
    lib, C = pkg.load_library(), pkg._cabi
    s = C.Shape()
    s.B, s.NH, s.S, s.DHQK, s.DHHV, s.chunk_size, s.dtype, s.impl = 1, NH, S, DK, DV, L, C.F32, C.IMPL_AUTO
    per_state = NH * DK * DV * 4
    assert lib.mlstm_b200_workspace_bytes(ctypes.byref(s), 0) >= (S // 32 + 1) * per_state
    assert NH * (S // 32 + 1) * DK * DV > 2 ** 31
    one = O.make_inputs(1, 1, S, DK, DV, seed=4, dtype=torch.float32)
    gen = torch.Generator(device="cuda").manual_seed(4)
    t = {}
    for name, x in one.items():
        shape = (1, NH) + tuple(x.shape[2:])
        y = torch.randn(shape, device="cuda", generator=gen) + (3.0 if name == "f" else 0.0)
        y[:, 0] = x[:, 0].cuda()
        y[:, NH - 1] = x[:, 0].cuda()
        t[name] = y
    got, _, launches = _fwbw(pkg, t, L)
    assert launches == (2, 4)
    for name, x in got.items():
        assert torch.equal(x[:, 0], x[:, NH - 1]), name
    first = {k: v[:, :1] for k, v in got.items()}
    del got, t
    torch.cuda.empty_cache()
    _assert_close(first, _oracle(one, torch.float32, L), F32_TOL, "first head of the large call")


def test_compile_fullgraph_bit_identical(pkg):
    """torch.compile(fullgraph=True) of the fp32 (256, 512) drop-in (with states) is bit-identical to eager."""
    torch._dynamo.reset()
    DK, DV, B, NH, S = 256, 512, 1, 2, 192
    g = torch.Generator().manual_seed(3)
    mk = lambda *s, sc=1.0, sh=0.0: (torch.randn(*s, generator=g) * sc + sh).cuda().requires_grad_(True)  # noqa: E731
    ts = [mk(B, NH, S, DK), mk(B, NH, S, DK), mk(B, NH, S, DV), mk(B, NH, S, sc=0.5), mk(B, NH, S, sh=3.0),
          mk(B, NH, DK, DV, sc=0.1), mk(B, NH, DK, sc=0.1), mk(B, NH, 1)]

    def fn(q, k, v, i, f, c0, n0, m0):
        h, (c, n, m) = pkg.mlstm_chunkwise__b200(q, k, v, i, f, c_initial=c0, n_initial=n0, m_initial=m0, chunk_size=64,
                                                 return_last_states=True)
        return h, c

    douts = [torch.randn(B, NH, S, DV, device="cuda"), torch.randn(B, NH, DK, DV, device="cuda")]

    def run(f_):
        for x in ts:
            x.grad = None
        outs = f_(*ts)
        torch.autograd.backward(outs, douts)
        return [o.detach().clone() for o in outs] + [x.grad.clone() for x in ts if x.grad is not None]

    eager = run(fn)
    compiled = run(torch.compile(fn, fullgraph=True))
    torch._dynamo.reset()
    assert len(eager) == len(compiled)
    for x, y in zip(eager, compiled):
        assert x.dtype == y.dtype and torch.equal(x, y)


def test_refusal_names_the_limits(pkg):
    B, NH, S = 1, 1, 64
    q, k, v = (torch.randn(B, NH, S, 512, device="cuda") for _ in range(3))
    i, f = torch.randn(B, NH, S, device="cuda"), torch.randn(B, NH, S, device="cuda")
    with pytest.raises(RuntimeError, match="DHQK <= 256 and DHHV <= 512"):
        pkg.mlstm_chunkwise__b200(q, k, v, i, f, chunk_size=64)
