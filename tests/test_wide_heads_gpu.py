"""xLSTM-Large's head geometry (DHQK, DHHV) = (256, 512) on the tensor-core route: the forward is tc_fw_wide (eight
64-wide column blocks of v / h / C per head in one launch), the backward 4 x 8 tc_bw<64> block problems whose dq / dk /
dv partials are summed in-kernel (TMA reduce-add stores) and whose 32 di / df partials are summed in fp32 by one more
kernel, the recurrent kernels a column-split k_recurrent.  Everything is measured against the float64 oracle at the 16-bit bar (max|a-b| / max|b| per
tensor < 2e-2) on inputs rounded to the test dtype; B * NH <= 2 and S <= 512 keep the oracle cheap."""
import ctypes
import os
import sys

import pytest
import torch

from oracle import mlstm_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import unnormalized_oracle as U  # noqa: E402

pytestmark = pytest.mark.gpu
DK, DV = 256, 512
DTYPES = [torch.bfloat16, torch.float16]
DTYPE_IDS = ["bf16", "fp16"]
SEQ = ("q", "k", "v", "i", "f", "dh")
MODES = [0, 1, 2]  # C-ABI siging: exponential input gate, sigmoid input gate, sigmoid input gate without normaliser
MODE_IDS = ["exp", "siging", "siging_unnorm"]


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as G

    G.build()
    import xlstm_yolo_clean_b200 as p

    return p


def _inputs(B, NH, S, seed, states, mode=0):
    inp = O.make_inputs(B, NH, S, DK, DV, seed=seed, dtype=torch.float32, with_states=states)
    if states and mode:  # the sigmoid-input-gate cell has no max state
        inp["m0"] = torch.zeros_like(inp["m0"])
    return inp


def _api(mode):
    return dict(siging=mode != 0, normalize=mode != 2)


def _fwbw(pkg, t, L, reverse=False, mode=0, states=False, save_states=True, grad_dtype=None):
    kw = dict(c_initial=t["c0"], n_initial=t["n0"], m_initial=t["m0"]) if states else {}
    h, n_out, m_out, last, cst = pkg.mlstm_chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=L,
                                                        return_last_states=states, reverse=reverse,
                                                        save_states=save_states, **_api(mode), **kw)
    n_fw = pkg.last_launch_count()
    g = pkg.mlstm_chunkwise_bw(t["q"], t["k"], t["v"], t["i"], t["f"], n_out, m_out, t["dh"], chunk_size=L, c_states=cst,
                               reverse=reverse, dc_last=t["dc_last"] if states else None, want_dc_initial=states,
                               grad_dtype=grad_dtype, **_api(mode), **kw)
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


def _tensor_route(pkg):
    pkg.set_default_impl("tensor")
    return pkg


@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("reverse", [False, True], ids=["causal", "anticausal"])
@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
def test_wide_parity_with_states(pkg, dtype, reverse, mode):
    """h, dq, dk, dv, di, df, the last states and dC_initial -- with initial states and dC_last -- at a ragged S (196 =
    one full and one 68-token tile), with the forward's saved block states."""
    S, L = 196, 4
    assert pkg.tensor_path_supported(1, 2, S, DK, DV, dtype, chunk_size=L)
    inp = _inputs(1, 2, S, seed=3 + 7 * reverse + 3 * mode, states=True, mode=mode)
    t = {k: v.to(dtype).cuda() for k, v in inp.items()}
    _tensor_route(pkg)
    try:
        got, cst, (n_fw, _) = _fwbw(pkg, t, L, reverse, mode, states=True)
    finally:
        pkg.set_default_impl("auto")
    assert cst is not None and n_fw == 1
    want = _oracle(inp, dtype, L, reverse, mode, states=True)
    _assert_close(got, want, 2e-2, f"(256, 512) {dtype} reverse={reverse} siging={mode}")


@pytest.mark.parametrize("reverse", [False, True], ids=["causal", "anticausal"])
@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
def test_wide_parity_over_four_tiles_plain(pkg, dtype, reverse):
    """No states, S = 452 (three full tiles and a ragged fourth): the C / n carry across tiles."""
    S, L = 452, 4
    inp = _inputs(1, 2, S, seed=41 + reverse, states=False)
    t = {k: v.to(dtype).cuda() for k, v in inp.items()}
    got, _, _ = _fwbw(pkg, t, L, reverse)
    _assert_close(got, _oracle(inp, dtype, L, reverse), 2e-2, f"(256, 512) {dtype} S=452")


def test_wide_strided_bshd_views(pkg):
    """xLSTM-Large's layout: q / k / v are (B, S, NH, D) projections transposed to (B, NH, S, D) views, taken as they are."""
    dtype, S = torch.bfloat16, 384
    inp = _inputs(1, 2, S, seed=90, states=False)
    t = {}
    for name, x in inp.items():
        x = x.to(dtype).cuda()
        t[name] = x.transpose(1, 2).contiguous().transpose(1, 2) if name in ("q", "k", "v", "dh") else x
    assert not t["q"].is_contiguous() and not t["v"].is_contiguous()
    got, _, _ = _fwbw(pkg, t, 64)
    _assert_close(got, _oracle(inp, dtype, 64), 2e-2, "strided (256, 512)")


@pytest.mark.parametrize("reverse", [False, True], ids=["causal", "anticausal"])
def test_wide_in_kernel_soft_cap(pkg, reverse):
    """gate_soft_cap: the outputs of the oracle fed with capped gates, dI / dF w.r.t. the pre-activations."""
    cap, S = 15.0, 200
    g = torch.Generator().manual_seed(S + reverse)
    dt = torch.bfloat16
    q, k = (torch.randn(1, 2, S, DK, generator=g).to(dt).cuda() for _ in range(2))
    v, dh = (torch.randn(1, 2, S, DV, generator=g).to(dt).cuda() for _ in range(2))
    pre_i = (-6.0 + torch.randn(1, 2, S, generator=g)).to(dt).cuda()
    pre_f = (6.0 + 2.0 * torch.randn(1, 2, S, generator=g)).to(dt).cuda()
    h, n_out, m_out, _, cst = pkg.mlstm_chunkwise_fw(q, k, v, pre_i, pre_f, chunk_size=4, reverse=reverse, gate_soft_cap=cap)
    dq, dk, dv, di, df, _ = pkg.mlstm_chunkwise_bw(q, k, v, pre_i, pre_f, n_out, m_out, dh, chunk_size=4, c_states=cst,
                                                   reverse=reverse, gate_soft_cap=cap)
    torch.cuda.synchronize()
    ti, tf = torch.tanh(pre_i.double().cpu() / cap), torch.tanh(pre_f.double().cpu() / cap)
    seq = (lambda x: x.flip(2)) if reverse else (lambda x: x)
    r = [seq(x.double().cpu()) for x in (q, k, v)] + [seq(cap * ti), seq(cap * tf), seq(dh.double().cpu())]
    h_ref, _, grads = O.fwbw(*r, chunk_size=4)
    want = dict(h=h_ref, dq=grads[0], dk=grads[1], dv=grads[2], di=grads[3] * seq(1 - ti ** 2), df=grads[4] * seq(1 - tf ** 2))
    got = dict(h=h, dq=dq, dk=dk, dv=dv, di=di, df=df)
    for name in want:
        assert O.rel_err(seq(got[name].double().cpu()), want[name]) < 2e-2, name


def test_wide_fp16_gradients_from_the_bf16_kernel(pkg):
    """grad_dtype: the reduce-add stores of the later block problems add into fp16 gradients of a bf16 call.  The bf16
    gradients carry one bf16 rounding per partial sum (dq / dk 8, dv 4), so the two differ by more than
    the single rounding of the rectangular pairs; both are within the 16-bit bar of the oracle."""
    S = 200
    inp = _inputs(1, 2, S, seed=71, states=False)
    t = {k: v.to(torch.bfloat16).cuda() for k, v in inp.items()}
    base, _, _ = _fwbw(pkg, t, 8)
    got, _, _ = _fwbw(pkg, t, 8, grad_dtype=torch.float16)
    want = _oracle(inp, torch.bfloat16, 8)
    for name in ("dq", "dk", "dv", "di", "df"):
        assert got[name].dtype == torch.float16 and base[name].dtype == torch.bfloat16
        assert O.rel_err(got[name].double().cpu(), base[name].double().cpu()) < 1.2e-2, name
        assert O.rel_err(got[name].double().cpu(), want[name]) < 2e-2, name
        assert O.rel_err(base[name].double().cpu(), want[name]) < 2e-2, name


def test_wide_launch_counts_saved_vs_recomputed_and_repeatable(pkg):
    """Forward: one launch.  Backward: one launch per block problem (32) with the forward's saved states, plus the fp32
    sum of the di / df partials (1); without them every block problem first recomputes its slice of the states (64 + 1).
    With initial states and dC_last / dC_initial each
    problem also gathers its dC_last block and scatters its dC_initial block (+ 64); recomputing, it gathers its C_0 / n_0
    blocks as well (+ 64).  Repeated calls are bit-identical.  Saved and recomputed states agree to the 16-bit rounding of
    the state operand: tc_fw_wide accumulates K^T (abar.V) with abar.V rounded, the square recompute (abar.K)^T V with
    abar.K rounded, so the two differ in the last bit of some state entries."""
    inp = _inputs(1, 2, 324, seed=5, states=True)
    t = {k: v.to(torch.bfloat16).cuda() for k, v in inp.items()}
    _tensor_route(pkg)
    try:
        h, n_out, m_out, _, cst = pkg.mlstm_chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=4)
        assert pkg.last_launch_count() == 1 and cst is not None
        h2, _, _, _, cst2 = pkg.mlstm_chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=4)
        assert torch.equal(cst, cst2)
        args = (t["q"], t["k"], t["v"], t["i"], t["f"], n_out, m_out, t["dh"])
        a = pkg.mlstm_chunkwise_bw(*args, chunk_size=4, c_states=cst)
        assert pkg.last_launch_count() == 32 + 1
        b = pkg.mlstm_chunkwise_bw(*args, chunk_size=4, c_states=None)
        assert pkg.last_launch_count() == 64 + 1
        c = pkg.mlstm_chunkwise_bw(*args, chunk_size=4, c_states=cst2)
        kw = dict(c_initial=t["c0"], n_initial=t["n0"], m_initial=t["m0"])
        _, n_out, m_out, _, cst = pkg.mlstm_chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=4, **kw)
        args = (t["q"], t["k"], t["v"], t["i"], t["f"], n_out, m_out, t["dh"])
        d = pkg.mlstm_chunkwise_bw(*args, chunk_size=4, c_states=cst, dc_last=t["dc_last"], want_dc_initial=True, **kw)
        assert pkg.last_launch_count() == 32 + 2 * 32 + 1
        d2 = pkg.mlstm_chunkwise_bw(*args, chunk_size=4, c_states=cst, dc_last=t["dc_last"], want_dc_initial=True, **kw)
        e = pkg.mlstm_chunkwise_bw(*args, chunk_size=4, c_states=None, dc_last=t["dc_last"], want_dc_initial=True, **kw)
        assert pkg.last_launch_count() == 64 + 4 * 32 + 1
    finally:
        pkg.set_default_impl("auto")
    torch.cuda.synchronize()
    assert torch.equal(h, h2)
    for x, y, z in zip(a[:5], b[:5], c[:5]):
        assert torch.equal(x, z) and O.rel_err(y, x) < 2e-2
    for x, y, z in zip(d, e, d2):
        assert torch.equal(x, z) and O.rel_err(y, x) < 2e-2


def test_wide_dropin_under_fp16_autocast(pkg):
    """mlstm_chunkwise__b200 under fp16 autocast with the bf16 kernel dtype (custom_fwd(cast_inputs=bf16)): bf16 h, fp16
    gradients written by the kernel, both within the bar of the oracle on the bf16-rounded inputs."""
    S = 256
    inp = _inputs(1, 2, S, seed=13, states=False)
    ts = [inp[n].to(torch.float16).cuda().requires_grad_(True) for n in ("q", "k", "v", "i", "f")]
    with torch.autocast("cuda", dtype=torch.float16):
        h = pkg.mlstm_chunkwise__b200(*ts, chunk_size=64)
    dh = inp["dh"].to(torch.bfloat16).cuda()
    h.backward(dh)
    torch.cuda.synchronize()
    assert h.dtype == torch.bfloat16 and all(x.grad.dtype == torch.float16 for x in ts)
    r = {k: v.to(torch.float16).to(torch.bfloat16).double() for k, v in inp.items()}
    h_ref, _, g = O.fwbw(r["q"], r["k"], r["v"], r["i"], r["f"], r["dh"], chunk_size=64)
    assert O.rel_err(h.double().cpu(), h_ref) < 2e-2
    for x, w, name in zip(ts, g, ("dq", "dk", "dv", "di", "df")):
        assert O.rel_err(x.grad.double().cpu(), w) < 2e-2, name


def test_wide_fused_epilogue_is_refused(pkg):
    """The fused cell-output epilogue does not exist at (256, 512): the call fails instead of running something else."""
    from xlstm_yolo_clean_b200 import backend

    B, NH, S = 1, 2, 128
    q, k = (torch.randn(B, NH, S, DK, device="cuda", dtype=torch.bfloat16) for _ in range(2))
    v = torch.randn(B, NH, S, DV, device="cuda", dtype=torch.bfloat16)
    i, f = torch.randn(B, NH, S, device="cuda", dtype=torch.bfloat16), torch.randn(B, NH, S, device="cuda", dtype=torch.bfloat16)
    y = torch.empty(B, S, NH, DV, device="cuda", dtype=torch.bfloat16).transpose(1, 2)
    w = torch.ones(NH * DV, device="cuda")
    epi = backend.FwEpilogue(y, None, w, None, None, 1e-5, False)
    with pytest.raises(RuntimeError, match="epilogue"):
        backend._fw_launch(q, k, v, i, f, None, None, None, None, False, 64, 1e-6, None, False, False, False, 0.0, epi)
    lib = pkg.load_library()
    s = pkg._cabi.Shape()
    s.B, s.NH, s.S, s.DHQK, s.DHHV, s.chunk_size, s.dtype = B, NH, S, DK, DV, 64, pkg._cabi.BF16
    assert lib.mlstm_b200_debug_fw_epilogue_clusters(ctypes.byref(s)) == 0


def test_wide_compile_fullgraph_bit_identical_and_opcheck(pkg):
    """torch.compile(fullgraph=True) of the drop-in (with states) is bit-identical to eager, and opcheck passes for the
    forward and backward ops at this pair."""
    torch._dynamo.reset()
    B, NH, S = 1, 2, 192
    g = torch.Generator().manual_seed(3)
    dev = "cuda"
    mk = lambda *s, sc=1.0, sh=0.0: (torch.randn(*s, generator=g) * sc + sh).to(dev, torch.bfloat16).requires_grad_(True)  # noqa: E731
    ts = [mk(B, NH, S, DK), mk(B, NH, S, DK), mk(B, NH, S, DV), mk(B, NH, S, sc=0.5), mk(B, NH, S, sh=3.0),
          (torch.randn(B, NH, DK, DV, generator=g) * 0.1).to(dev).requires_grad_(True),
          (torch.randn(B, NH, DK, generator=g) * 0.1).to(dev).requires_grad_(True),
          torch.randn(B, NH, 1, generator=g).to(dev).requires_grad_(True)]

    def fn(q, k, v, i, f, c0, n0, m0):
        h, (c, n, m) = pkg.mlstm_chunkwise__b200(q, k, v, i, f, c_initial=c0, n_initial=n0, m_initial=m0, chunk_size=64,
                                                 return_last_states=True)
        return h, c

    douts = [torch.randn(B, NH, S, DV, device=dev, dtype=torch.bfloat16), torch.randn(B, NH, DK, DV, device=dev)]

    def run(f_):
        for t in ts:
            t.grad = None
        outs = f_(*ts)
        torch.autograd.backward(outs, douts)
        return [o.detach().clone() for o in outs] + [t.grad.clone() for t in ts]

    eager = run(fn)
    compiled = run(torch.compile(fn, fullgraph=True))
    for x, y in zip(eager, compiled):
        assert x.dtype == y.dtype and torch.equal(x, y)
    torch._dynamo.reset()
    ops = torch.ops.mlstm_b200
    q, k, v, i, f = (t.detach().requires_grad_(True) for t in ts[:5])
    fw_args = (q, k, v, i, f, None, None, None, None, None, True, 64, 1e-6, 0, True, False, False, 0.0, None)
    torch.library.opcheck(ops.chunkwise_fw, fw_args)
    h, nm, _, _, _, cs = (t.detach() for t in ops.chunkwise_fw(*fw_args))
    qd, kd, vd, idd, fd = (t.detach() for t in (q, k, v, i, f))
    torch.library.opcheck(ops.chunkwise_bw, (qd, kd, vd, idd, fd, nm[0], nm[1], torch.randn_like(h), None, None, None, None,
                                             cs, None, None, 64, 1e-6, 0, False, False, False, 0.0, torch.float16))
    torch.library.opcheck(ops.recurrent_sequence, (qd[:, :, :8], kd[:, :, :8], vd[:, :, :8], idd[:, :, :8], fd[:, :, :8],
                                                   None, None, None, True, 1e-6, False))


# ------------------------------------------------------------------------------------------------ recurrent kernels
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-5), (torch.bfloat16, 2e-2), (torch.float16, 2e-2)],
                         ids=["fp32", "bf16", "fp16"])
def test_wide_recurrent_sequence_matches_step_recurrence(pkg, dtype, tol, mode):
    S = 24
    inp = O.make_inputs(1, 2, S, DK, DV, seed=11 + mode, dtype=torch.float32, with_states=True)
    if mode:
        inp["m0"] = torch.zeros_like(inp["m0"])
    r = {k: v.to(dtype).double() for k, v in inp.items()}
    if mode == 0:
        h_ref, (c_ref, n_ref, m_ref) = O.step_recurrence(r["q"], r["k"], r["v"], r["i"], r["f"], r["c0"], r["n0"], r["m0"])
    elif mode == 1:
        h_ref, _, _, (c_ref, n_ref, m_ref), _ = O.chunkwise_fw(r["q"], r["k"], r["v"], r["i"], r["f"], r["c0"], r["n0"], None,
                                                               chunk_size=1, siging=True)
    else:
        h_ref, _, _, (c_ref, n_ref, m_ref) = U.chunkwise_fw(r["q"], r["k"], r["v"], r["i"], r["f"], r["c0"], r["n0"],
                                                            chunk_size=1)
    t = {k: v.to(dtype).cuda() for k, v in inp.items()}
    h, (c, n, m) = pkg.mlstm_recurrent_sequence__b200(t["q"], t["k"], t["v"], t["i"], t["f"], t["c0"], t["n0"],
                                                      t["m0"], return_last_states=True,
                                                      siging=mode != 0, normalize=mode != 2)
    assert pkg.last_launch_count() == 1
    torch.cuda.synchronize()
    assert h.shape == (1, 2, S, DV) and c.shape == (1, 2, DK, DV)
    for name, a, b in (("h", h, h_ref), ("c", c, c_ref), ("n", n, n_ref), ("m", m, m_ref)):
        assert O.rel_err(a.double().cpu().reshape(b.shape), b) < tol, name


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
def test_wide_chunkwise_prefix_continued_by_the_sequence_kernel(pkg, dtype):
    """A return_last_states chunkwise call over the first 256 tokens, continued by mlstm_recurrent_sequence__b200 over
    the last 60 from its (C, n, m), gives what one chunkwise call over all 316 tokens gives."""
    S0, S1 = 256, 60
    inp = O.make_inputs(1, 2, S0 + S1, DK, DV, seed=17, dtype=torch.float32)
    t = {k: v.to(dtype).cuda() for k, v in inp.items()}
    full = pkg.mlstm_chunkwise__b200(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=4)
    pre = {k: t[k][:, :, :S0] for k in ("q", "k", "v", "i", "f")}
    post = {k: t[k][:, :, S0:] for k in ("q", "k", "v", "i", "f")}
    h0, (c, n, m) = pkg.mlstm_chunkwise__b200(pre["q"], pre["k"], pre["v"], pre["i"], pre["f"], chunk_size=64,
                                              return_last_states=True)
    h1 = pkg.mlstm_recurrent_sequence__b200(post["q"], post["k"], post["v"], post["i"], post["f"], c, n, m)
    torch.cuda.synchronize()
    assert O.rel_err(torch.cat([h0, h1], 2).double().cpu(), full.double().cpu()) < 2e-2
    assert torch.equal(h0, full[:, :, :S0])
