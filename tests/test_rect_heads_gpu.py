"""Rectangular heads (DHQK, DHHV) = (32, 64) and (64, 128) in bf16 / fp16 on the tensor-core route: the forward runs
both D-wide column blocks of v / h / C in one launch (tc_fw_rect), the backward runs as two square tc_bw<DHQK> block
problems whose dq / dk (TMA reduce-add stores) and di / df (owner-thread accumulate) partials are summed in-kernel --
at DHQK = 32 that is the only place the accumulate flags of tc_bw<32> run.  Everything is measured against the float64
oracle at the 16-bit bar (max|a-b| / max|b| per tensor < 2e-2), plus the recurrent kernels at the same pairs."""
import math
import os
import sys

import pytest
import torch

from oracle import mlstm_oracle as O

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "baseline", "_ref")
needs_ref = pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "mlstm_kernels")),
                               reason="reference not staged under baseline/_ref (tools/stage_reference.sh)")

PAIRS = [(32, 64), (64, 128)]
PAIR_IDS = ["qk32_v64", "qk64_v128"]
DTYPES = [torch.bfloat16, torch.float16]
DTYPE_IDS = ["bf16", "fp16"]
SEQ = ("q", "k", "v", "i", "f", "dh")


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as G

    G.build()
    import xlstm_yolo_clean_b200 as p

    return p


def _inputs(B, NH, S, DK, DV, seed, states, siging):
    inp = O.make_inputs(B, NH, S, DK, DV, seed=seed, dtype=torch.float32, with_states=states)
    if states and siging:  # the sigmoid-input-gate cell has no max state
        inp["m0"] = torch.zeros_like(inp["m0"])
    return inp


def _bshd(t, dt):
    """q / k as the two halves of one (B, S, NH, 2 DK) tensor, v with its own (B, S, NH, DV) token stride."""
    B, NH, S, DK = t["q"].shape
    qk = torch.empty(B, S, NH, 2 * DK, dtype=dt, device="cuda")
    qk[..., :DK] = t["q"].transpose(1, 2)
    qk[..., DK:] = t["k"].transpose(1, 2)
    out = dict(t)
    out["q"], out["k"] = qk[..., :DK].transpose(1, 2), qk[..., DK:].transpose(1, 2)
    out["v"] = t["v"].transpose(1, 2).contiguous().transpose(1, 2)
    assert not out["q"].is_contiguous() and not out["v"].is_contiguous()
    return out


def _fwbw(pkg, t, L, reverse=False, siging=False, states=False, save_states=True, grad_dtype=None):
    kw = dict(c_initial=t["c0"], n_initial=t["n0"], m_initial=t["m0"]) if states else {}
    h, n_out, m_out, last, cst = pkg.mlstm_chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=L,
                                                        return_last_states=states, reverse=reverse, siging=siging,
                                                        save_states=save_states, **kw)
    n_fw = pkg.last_launch_count()
    g = pkg.mlstm_chunkwise_bw(t["q"], t["k"], t["v"], t["i"], t["f"], n_out, m_out, t["dh"], chunk_size=L, c_states=cst,
                               reverse=reverse, siging=siging, dc_last=t["dc_last"] if states else None,
                               want_dc_initial=states, grad_dtype=grad_dtype, **kw)
    n_bw = pkg.last_launch_count()
    torch.cuda.synchronize()
    out = dict(h=h, dq=g[0], dk=g[1], dv=g[2], di=g[3], df=g[4])
    if states:
        out.update(c_last=last[0], n_last=last[1], m_last=last[2], dc0=g[5])
    return out, cst, (n_fw, n_bw)


def _oracle(inp, dtype, L, reverse=False, siging=False, states=False):
    r = {k: v.to(dtype).double() for k, v in inp.items()}
    if reverse:
        r = {k: (v.flip(2) if k in SEQ else v) for k, v in r.items()}
    st = (r["c0"], r["n0"], r["m0"]) if states else (None, None, None)
    h, last, g = O.fwbw(r["q"], r["k"], r["v"], r["i"], r["f"], r["dh"], *st, dc_last=r["dc_last"] if states else None,
                        chunk_size=L, siging=siging)
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


@pytest.mark.parametrize("states", [False, True], ids=["plain", "states"])
@pytest.mark.parametrize("siging", [False, True], ids=["exp", "siging"])
@pytest.mark.parametrize("reverse", [False, True], ids=["causal", "anticausal"])
@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_rect_parity(pkg, DK, DV, dtype, reverse, siging, states):
    """h, dq, dk, dv, di, df -- with initial states and dC_last also the last states and dC_initial -- at a ragged S
    (196 = one full and one 68-token tile), on the tensor route with the forward's saved block states."""
    S, L = 196, 4
    assert pkg.tensor_path_supported(2, 2, S, DK, DV, dtype, chunk_size=L)
    inp = _inputs(2, 2, S, DK, DV, seed=DK + 7 * reverse + 3 * siging, states=states, siging=siging)
    t = {k: v.to(dtype).cuda() for k, v in inp.items()}
    pkg.set_default_impl("tensor")
    try:
        got, cst, _ = _fwbw(pkg, t, L, reverse, siging, states)
    finally:
        pkg.set_default_impl("auto")
    assert cst is not None
    _assert_close(got, _oracle(inp, dtype, L, reverse, siging, states), 2e-2, f"({DK}, {DV}) {dtype}")


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_rect_strided_bshd_views(pkg, DK, DV, dtype):
    """q / k as the two halves of one (B, S, NH, 2 DHQK) tensor and v with its own token stride, taken as they are."""
    inp = _inputs(2, 3, 256, DK, DV, seed=90 + DK, states=False, siging=False)
    t = _bshd({k: v.to(dtype).cuda() for k, v in inp.items()}, dtype)
    pkg.set_default_impl("tensor")
    try:
        got, _, _ = _fwbw(pkg, t, 64)
    finally:
        pkg.set_default_impl("auto")
    _assert_close(got, _oracle(inp, dtype, 64), 2e-2, f"strided ({DK}, {DV}) {dtype}")


@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_rect_launch_counts_and_recompute(pkg, DK, DV):
    """Forward: one launch.  Backward: one launch per block problem (two) with the forward's saved states; without them
    every block problem first recomputes its slice of the states (a square forward), so four.  Both backward forms, and
    two identical calls, agree bit for bit."""
    inp = _inputs(2, 2, 324, DK, DV, seed=5, states=True, siging=False)
    t = {k: v.to(torch.bfloat16).cuda() for k, v in inp.items()}
    pkg.set_default_impl("tensor")
    try:
        h, n_out, m_out, _, cst = pkg.mlstm_chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=4)
        assert pkg.last_launch_count() == 1 and cst is not None
        h2, _, _, _, cst2 = pkg.mlstm_chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=4)
        args = (t["q"], t["k"], t["v"], t["i"], t["f"], n_out, m_out, t["dh"])
        a = pkg.mlstm_chunkwise_bw(*args, chunk_size=4, c_states=cst)
        assert pkg.last_launch_count() == 2
        b = pkg.mlstm_chunkwise_bw(*args, chunk_size=4, c_states=None)
        assert pkg.last_launch_count() == 4
        c = pkg.mlstm_chunkwise_bw(*args, chunk_size=4, c_states=cst2)
        # with initial states, dC_last and dC_initial: per-block copies of C_0 (recompute only), dC_last and dC_initial
        kw = dict(c_initial=t["c0"], n_initial=t["n0"], m_initial=t["m0"])
        _, n_out, m_out, _, cst = pkg.mlstm_chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=4, **kw)
        args = (t["q"], t["k"], t["v"], t["i"], t["f"], n_out, m_out, t["dh"])
        d = pkg.mlstm_chunkwise_bw(*args, chunk_size=4, c_states=cst, dc_last=t["dc_last"], want_dc_initial=True, **kw)
        assert pkg.last_launch_count() == 2 + 2 + 2
        e = pkg.mlstm_chunkwise_bw(*args, chunk_size=4, c_states=None, dc_last=t["dc_last"], want_dc_initial=True, **kw)
        assert pkg.last_launch_count() == 4 + 2 * 2 + 2 + 2
    finally:
        pkg.set_default_impl("auto")
    torch.cuda.synchronize()
    assert torch.equal(h, h2)
    for x, y, z in zip(a[:5], b[:5], c[:5]):
        assert torch.equal(x, y) and torch.equal(x, z)
    for x, y in zip(d, e):
        assert torch.equal(x, y)


@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_rect_tensor_route_agrees_with_exact_route(pkg, DK, DV):
    """The same bf16 call through the fp32 FFMA kernels (the route rectangular heads took before) and the tensor route."""
    inp = _inputs(2, 3, 384, DK, DV, seed=11, states=True, siging=False)
    t = {k: v.to(torch.bfloat16).cuda() for k, v in inp.items()}
    pkg.set_default_impl("exact")
    try:
        ex, _, (fw_ex, _) = _fwbw(pkg, t, 64, states=True)
    finally:
        pkg.set_default_impl("auto")
    tc, _, (fw_tc, _) = _fwbw(pkg, t, 64, states=True)
    assert fw_tc == 1 and fw_ex != 1  # AUTO took the tensor route, EXACT the FFMA kernels
    for k in tc:
        assert O.rel_err(tc[k].double().cpu(), ex[k].double().cpu()) < 2e-2, k


@pytest.mark.parametrize("siging", [False, True], ids=["exp", "siging"])
@pytest.mark.parametrize("reverse", [False, True], ids=["causal", "anticausal"])
@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_rect_in_kernel_soft_cap_equals_capping_first(pkg, DK, DV, reverse, siging):
    """gate_soft_cap at rectangular heads: same outputs as the fp64 oracle fed with capped gates, and dI / dF w.r.t. the
    pre-activations (chain rule through cap * tanh(x / cap))."""
    cap, S = 15.0, 200
    g = torch.Generator().manual_seed(DK + S)
    dt = torch.bfloat16
    q, k = (torch.randn(2, 3, S, DK, generator=g).to(dt).cuda() for _ in range(2))
    v, dh = (torch.randn(2, 3, S, DV, generator=g).to(dt).cuda() for _ in range(2))
    pre_i = (-6.0 + torch.randn(2, 3, S, generator=g)).to(dt).cuda()
    pre_f = (6.0 + 2.0 * torch.randn(2, 3, S, generator=g)).to(dt).cuda()
    h, n_out, m_out, _, cst = pkg.mlstm_chunkwise_fw(q, k, v, pre_i, pre_f, chunk_size=4, reverse=reverse, siging=siging,
                                                     gate_soft_cap=cap)
    dq, dk, dv, di, df, _ = pkg.mlstm_chunkwise_bw(q, k, v, pre_i, pre_f, n_out, m_out, dh, chunk_size=4, c_states=cst,
                                                   reverse=reverse, siging=siging, gate_soft_cap=cap)
    torch.cuda.synchronize()
    ci = cap * torch.tanh(pre_i.double().cpu() / cap)
    cf = cap * torch.tanh(pre_f.double().cpu() / cap)
    seq = (lambda x: x.flip(2)) if reverse else (lambda x: x)
    r = [seq(x.double().cpu()) for x in (q, k, v)] + [seq(ci), seq(cf), seq(dh.double().cpu())]
    h_ref, _, grads = O.fwbw(*r, chunk_size=4, siging=siging)
    want = dict(h=h_ref, dq=grads[0], dk=grads[1], dv=grads[2],
                di=grads[3] * seq(1 - torch.tanh(pre_i.double().cpu() / cap) ** 2),
                df=grads[4] * seq(1 - torch.tanh(pre_f.double().cpu() / cap) ** 2))
    got = dict(h=h, dq=dq, dk=dk, dv=dv, di=di, df=df)
    for name in want:
        assert O.rel_err(seq(got[name].double().cpu()), want[name]) < 2e-2, name


@pytest.mark.parametrize("kdt,gdt", [(torch.bfloat16, torch.float16), (torch.float16, torch.bfloat16)],
                         ids=["bf16_kernel_fp16_grads", "fp16_kernel_bf16_grads"])
@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_rect_gradients_in_the_callers_dtype(pkg, DK, DV, kdt, gdt):
    """grad_dtype at rectangular heads: the reduce-add stores of the second block problem add into gradients of the
    other 16-bit dtype; one rounding from the kernel-dtype gradients and within the 16-bit bar of the oracle."""
    S = 200
    inp = _inputs(2, 3, S, DK, DV, seed=71, states=False, siging=False)
    t = {k: v.to(kdt).cuda() for k, v in inp.items()}
    base, _, _ = _fwbw(pkg, t, math.gcd(S, 64))
    got, _, _ = _fwbw(pkg, t, math.gcd(S, 64), grad_dtype=gdt)
    want = _oracle(inp, kdt, math.gcd(S, 64))
    for name in ("dq", "dk", "dv", "di", "df"):
        assert got[name].dtype == gdt and base[name].dtype == kdt
        assert O.rel_err(got[name].double().cpu(), base[name].double().cpu()) < 6e-3, name
        assert O.rel_err(got[name].double().cpu(), want[name]) < 2e-2, name


# ------------------------------------------------------------------------------------------------ recurrent kernels
@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-5), (torch.bfloat16, 2e-2)], ids=["fp32", "bf16"])
@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_rect_recurrent_sequence_matches_step_recurrence(pkg, DK, DV, dtype, tol):
    inp = O.make_inputs(2, 3, 40, DK, DV, seed=11 + DK, dtype=torch.float32, with_states=True)
    r = {k: v.to(dtype).double() for k, v in inp.items()}
    h_ref, (c_ref, n_ref, m_ref) = O.step_recurrence(r["q"], r["k"], r["v"], r["i"], r["f"], r["c0"], r["n0"], r["m0"])
    t = {k: v.to(dtype).cuda() for k, v in inp.items()}
    h, (c, n, m) = pkg.mlstm_recurrent_sequence__b200(t["q"], t["k"], t["v"], t["i"], t["f"], t["c0"], t["n0"], t["m0"],
                                                      return_last_states=True)
    torch.cuda.synchronize()
    assert h.shape == (2, 3, 40, DV) and c.shape == (2, 3, DK, DV)
    for name, a, b in (("h", h, h_ref), ("c", c, c_ref), ("n", n, n_ref), ("m", m, m_ref)):
        assert O.rel_err(a.double().cpu().reshape(b.shape), b) < tol, name


@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_rect_step_kernel_chains_like_the_sequence(pkg, DK, DV):
    """Single steps fed with their own states reproduce one sequence call bit for bit (fp32)."""
    B, NH, S = 2, 4, 9
    g = torch.Generator().manual_seed(DK)
    q, k = (torch.randn(B, NH, S, DK, generator=g).cuda() for _ in range(2))
    v = torch.randn(B, NH, S, DV, generator=g).cuda()
    i, f = torch.randn(B, NH, S, generator=g).cuda(), (2 + torch.randn(B, NH, S, generator=g)).cuda()
    h_seq, (c_seq, n_seq, m_seq) = pkg.mlstm_recurrent_sequence__b200(q, k, v, i, f, return_last_states=True)
    c = torch.zeros(B, NH, DK, DV, device="cuda")
    n = torch.zeros(B, NH, DK, device="cuda")
    m = torch.zeros(B, NH, 1, device="cuda")
    hs = []
    for s in range(S):
        h, (c, n, m) = pkg.mlstm_recurrent_step__b200(q[:, :, s], k[:, :, s], v[:, :, s], i[:, :, s, None], f[:, :, s, None],
                                                       c, n, m)
        hs.append(h)
    torch.cuda.synchronize()
    assert torch.equal(torch.stack(hs, 2), h_seq) and torch.equal(c, c_seq) and torch.equal(n, n_seq)
    assert torch.equal(m, m_seq)


@needs_ref
@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_rect_behind_the_arbitrary_sequence_length_wrapper(pkg, DK, DV):
    """The reference's inference wrapper on a rectangular sequence whose length leaves a remainder: chained chunkwise
    calls hand (C, n) to each other and the B200 sequence kernel finishes the last tokens."""
    from functools import partial

    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import model_bench as MB

    MB._import_reference()
    from mlstm_kernels.torch.kernel_wrappers import wrap_chunkwise__arbitrary_sequence_length

    B, NH, S = 2, 3, 1003
    inp = O.make_inputs(B, NH, S, DK, DV, seed=S + DK, dtype=torch.float32)
    t = {k: v.to(torch.bfloat16).cuda() for k, v in inp.items()}
    h, states = wrap_chunkwise__arbitrary_sequence_length(
        mlstm_chunkwise_kernel=pkg.mlstm_siging_chunkwise__b200,
        mlstm_sequence_kernel=partial(pkg.mlstm_recurrent_sequence__b200, siging=True),
        mlstm_step_kernel=partial(pkg.mlstm_recurrent_step__b200, siging=True),
        q=t["q"], k=t["k"], v=t["v"], i=t["i"], f=t["f"], return_last_states=True, chunk_size=64, eps=1e-6,
        autocast_kernel_dtype=torch.bfloat16)
    torch.cuda.synchronize()
    d = {k: v.to(torch.bfloat16).double() for k, v in inp.items()}
    h_ref, _, _, last, _ = O.chunkwise_fw(d["q"], d["k"], d["v"], d["i"], d["f"], chunk_size=1, siging=True)
    assert h.shape == (B, NH, S, DV)
    assert O.rel_err(h.double().cpu(), h_ref) < 2e-2
    assert O.rel_err(states[0].double().cpu(), last[0]) < 2e-2 and O.rel_err(states[1].double().cpu(), last[1]) < 2e-2
