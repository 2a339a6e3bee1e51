"""Fused cell-output epilogue (mlstm_b200_fw_epilogue) for rectangular heads (DHQK, DHHV) = (32, 64) and (64, 128): the two
DHQK-wide column blocks of a head run in one two-CTA cluster and exchange the LayerNorm row statistics, so y is the
MultiHeadLayerNorm over the whole DHHV row.  Kernel level: the h written alongside y is bit-identical to the plain
rectangular forward's, and y equals the stand-alone cell-output kernel on that h (pinned to float64 group_norm in
test_cell_gpu.py) up to one rounding of the output dtype.  Cell level: mlstm_cell_b200 on a cell whose q / k are narrower
than v, one launch or two, against a float64 composition (oracle h -> per-head group_norm -> skip)."""
import pytest
import torch
import torch.nn.functional as F

from oracle import mlstm_oracle as O

pytestmark = pytest.mark.gpu

PAIRS = [(32, 64), (64, 128)]
PAIR_IDS = ["qk32_v64", "qk64_v128"]
KO_DTYPES = [(torch.bfloat16, torch.float16), (torch.float16, torch.float16), (torch.bfloat16, torch.bfloat16)]
KO_IDS = ["bf16_kernel_fp16_out", "fp16", "bf16"]


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as G

    G.build()
    import xlstm_yolo_clean_b200 as p

    return p


def rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def _tol(odt):
    return 2e-3 if odt == torch.float16 else 1.2e-2


def _layer_inputs(B, S, NH, DK, DV, kdt, odt, seed, v_scale=None):
    """qk (B, S, 2 NH DK), v (B, S, NH DV), gates (B, S, 2 NH) in the kernel dtype; x (B, S, NH DV) in the output dtype;
    fp32 LayerNorm weight / bias / skip.  ``v_scale`` = (scale, shift) of the second column half of every head's v."""
    g = torch.Generator().manual_seed(seed)
    dev = torch.device("cuda:0")
    qk = torch.randn(B, S, 2 * NH * DK, generator=g)
    v = torch.randn(B, S, NH, DV, generator=g)
    if v_scale is not None:
        v[..., DV // 2:] = v[..., DV // 2:] * v_scale[0] + v_scale[1]
    gates = torch.cat([torch.randn(B, S, NH, generator=g), 3 + torch.randn(B, S, NH, generator=g)], -1)
    x = torch.randn(B, S, NH * DV, generator=g)
    H = NH * DV
    par = ((1 + 0.1 * torch.randn(H, generator=g)).to(dev), (0.1 * torch.randn(H, generator=g)).to(dev),
           torch.randn(H, generator=g).to(dev))
    return (qk.to(kdt).to(dev), v.reshape(B, S, H).to(kdt).to(dev), gates.to(kdt).to(dev), x.to(odt).to(dev)) + par


def _fused(pkg, q, k, vv, i, f, y, x, w, b, sk, L, reverse, siging, cap, want_h, NH, DV):
    from xlstm_yolo_clean_b200 import backend

    B, S = y.shape[:2]
    heads = lambda t: t.view(B, S, NH, DV).transpose(1, 2)  # noqa: E731
    epi = backend.FwEpilogue(heads(y), None if x is None else heads(x), w, b, sk, 1e-5, want_h)
    h = backend._fw_launch(q, k, vv, i, f, None, None, None, None, False, L, 1e-6, None, want_h, reverse, siging, cap, epi)[0]
    return h, pkg.last_launch_count()


def _plain(pkg, q, k, vv, i, f, L, reverse, siging, cap):
    from xlstm_yolo_clean_b200 import backend

    return backend._fw_launch(q, k, vv, i, f, None, None, None, None, False, L, 1e-6, None, True, reverse, siging, cap)[0]


@pytest.mark.parametrize("siging", [False, True], ids=["exp", "siging"])
@pytest.mark.parametrize("reverse", [False, True], ids=["causal", "anticausal"])
@pytest.mark.parametrize("kdt,odt", KO_DTYPES, ids=KO_IDS)
@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_rect_epilogue_equals_kernel_plus_cell_out(pkg, DK, DV, kdt, odt, reverse, siging):
    B, S, NH, L = 2, 384, 4, 4
    qk, v, gates, x, w, b, sk = _layer_inputs(B, S, NH, DK, DV, kdt, odt, seed=DK + 3 * reverse + 5 * siging)
    q, k, vv, i, f = pkg.vil._heads(qk, v, gates, NH)
    assert q.shape[-1] == DK and vv.shape[-1] == DV
    h0 = _plain(pkg, q, k, vv, i, f, L, reverse, siging, 0.0)
    y = torch.empty(B, S, NH * DV, dtype=odt, device="cuda")
    h1, launches = _fused(pkg, q, k, vv, i, f, y, x, w, b, sk, L, reverse, siging, 0.0, True, NH, DV)
    torch.cuda.synchronize()
    assert launches == 1  # mLSTM forward, LayerNorm, relayout and skip in one kernel
    assert torch.equal(h1, h0)
    assert rel(y, pkg.cell_out(h0, w, b, sk, x, eps=1e-5, out_dtype=odt)) < _tol(odt)
    # inference flavour: no skip input, no bias, h not written
    y2 = torch.empty_like(y)
    h2, _ = _fused(pkg, q, k, vv, i, f, y2, None, w, None, None, L, reverse, siging, 0.0, False, NH, DV)
    torch.cuda.synchronize()
    assert h2 is None
    assert rel(y2, pkg.cell_out(h0, w, None, None, None, eps=1e-5, out_dtype=odt)) < _tol(odt)


@pytest.mark.parametrize("S", [100, 200])
@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_rect_epilogue_ragged_views_soft_cap_repeatable(pkg, DK, DV, S):
    """A ragged last tile (every row of it still takes part in the statistics exchange), y and x as (B, NH, S, DHHV)
    views of (B, S, NH DHHV) buffers with a larger token stride, the in-kernel gate soft cap, and bit-identical repeats."""
    B, NH, L, cap = 3, 4, 4, 15.0
    kdt, odt = torch.bfloat16, torch.float16
    qk, v, gates, x, w, b, sk = _layer_inputs(B, S, NH, DK, DV, kdt, odt, seed=S + DK)
    gates = gates * 8  # so that the cap matters
    q, k, vv, i, f = pkg.vil._heads(qk, v, gates, NH)
    H = NH * DV
    xbuf = torch.zeros(B, S, H + 64, dtype=odt, device="cuda")
    xbuf[..., :H] = x
    xs = xbuf[..., :H]
    outs = []
    for _ in range(2):
        ybuf = torch.full((B, S, H + 64), float("nan"), dtype=odt, device="cuda")
        y = ybuf[..., :H]
        h, launches = _fused(pkg, q, k, vv, i, f, y, xs, w, b, sk, L, False, False, cap, True, NH, DV)
        torch.cuda.synchronize()
        assert launches == 1
        assert torch.isnan(ybuf[..., H:]).all()  # nothing written outside the view
        outs.append((ybuf.clone(), h.clone()))
    assert torch.equal(outs[0][0][..., :H], outs[1][0][..., :H]) and torch.equal(outs[0][1], outs[1][1])
    h0 = _plain(pkg, q, k, vv, i, f, L, False, False, cap)
    assert torch.equal(outs[0][1], h0)
    assert rel(outs[0][0][..., :H], pkg.cell_out(h0, w, b, sk, x, eps=1e-5, out_dtype=odt)) < _tol(odt)


@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_rect_epilogue_statistics_span_both_column_blocks(pkg, DK, DV):
    """The second column half of every head's v scaled by 100 and shifted by 20: its h columns dwarf the first half's.
    LayerNorm over the whole DHHV row differs from a LayerNorm per DHQK-wide column block by O(1) in every element of the
    first half, so y only matches the row-wide reference if the two CTAs combined their statistics."""
    B, S, NH, L = 2, 256, 4, 4
    kdt, odt = torch.bfloat16, torch.float16
    qk, v, gates, x, w, b, sk = _layer_inputs(B, S, NH, DK, DV, kdt, odt, seed=11 * DK, v_scale=(100.0, 20.0))
    q, k, vv, i, f = pkg.vil._heads(qk, v, gates, NH)
    h0 = _plain(pkg, q, k, vv, i, f, L, False, False, 0.0)
    y = torch.empty(B, S, NH * DV, dtype=odt, device="cuda")
    _fused(pkg, q, k, vv, i, f, y, None, w, b, None, L, False, False, 0.0, False, NH, DV)
    torch.cuda.synchronize()
    want = pkg.cell_out(h0, w, b, None, None, eps=1e-5, out_dtype=odt)
    per_block = pkg.cell_out(h0.reshape(B, NH, S, 2, DK).transpose(2, 3).reshape(B, 2 * NH, S, DK),
                             w, b, None, None, eps=1e-5, out_dtype=odt)
    assert rel(per_block, want) > 0.1  # the case tells the two apart
    assert rel(y, want) < _tol(odt)


# ---------------------------------------------------------------------------------------------
class _Norm(torch.nn.Module):
    def __init__(self, H):
        super().__init__()
        self.weight = torch.nn.Parameter(0.1 * torch.randn(H))
        self.bias = torch.nn.Parameter(0.1 * torch.randn(H))
        self.eps = 1e-6

    @property
    def weight_proxy(self):
        return 1.0 + self.weight


class _RectCell(torch.nn.Module):
    """Attribute-compatible stand-in for MatrixLSTMCell (vision_lstm2.py:701-753) with q / k of width NH DHQK < NH DHHV."""

    def __init__(self, NH, DK, DV):
        super().__init__()
        Hqk, Hv = NH * DK, NH * DV
        self.dim, self.num_heads, self.gate_soft_cap = Hv, NH, 15.0
        self.use_autocast, self.autocast_dtype = True, torch.float16
        self.ifgate = torch.nn.Linear(2 * Hqk + Hv, 2 * NH)
        self.outnorm = _Norm(Hv)
        with torch.no_grad():
            self.ifgate.bias[:NH] = -2.0
            self.ifgate.bias[NH:] = torch.linspace(3.0, 6.0, NH)


class _OracleMlstm(torch.autograd.Function):
    """The oracle's chunkwise forward and its analytic backward (O.fwbw) as one differentiable float64 op."""

    @staticmethod
    def forward(ctx, q, k, v, i, f):
        ctx.save_for_backward(q, k, v, i, f)
        return O.chunkwise_fw(q, k, v, i, f, chunk_size=4, eps=1e-6)[0]

    @staticmethod
    def backward(ctx, dh):
        return tuple(O.fwbw(*ctx.saved_tensors, dh.contiguous(), chunk_size=4, eps=1e-6)[2][:5])


def _reference_cell(NH, cap, W, bb, ln_w, ln_b, ln_eps, qk, v, x, skip, reverse):
    """float64: ifgate + soft cap, the oracle's h on the fp16-rounded kernel inputs, group_norm per head over DHHV, skip.
    ``ln_w`` is the effective LayerNorm scale (weight_proxy)."""
    B, S, Hv = v.shape
    q, k = torch.chunk(qk, 2, -1)
    pre = F.linear(torch.cat([q, k, v], -1), W, bb)
    pre = cap * torch.tanh(pre / cap)
    r16 = lambda t: t + (t.to(torch.float16).double() - t).detach()  # noqa: E731  (kernel-dtype rounding, identity gradient)
    i, f = (r16(t).transpose(-1, -2) for t in torch.chunk(pre, 2, -1))
    qh, kh, vh = (r16(t).view(B, S, NH, -1).transpose(1, 2) for t in (q, k, v))
    if reverse:
        qh, kh, vh, i, f = (t.flip(2) for t in (qh, kh, vh, i, f))
    h = _OracleMlstm.apply(qh, kh, vh, i, f)
    if reverse:
        h = h.flip(2)
    DV = h.shape[-1]
    g = F.group_norm(h.transpose(1, 2).reshape(B * S, NH * DV), NH, ln_w, ln_b, ln_eps)
    return g.view(B, S, NH * DV) + skip * x


@pytest.mark.parametrize("reverse", [False, True], ids=["causal", "anticausal"])
@pytest.mark.parametrize("DK,DV", PAIRS, ids=PAIR_IDS)
def test_rect_cell_one_and_two_launches_match_float64(pkg, DK, DV, reverse):
    torch.manual_seed(DK + reverse)
    dev = torch.device("cuda:0")
    B, S, NH = 2, 196, 4
    Hqk, Hv = NH * DK, NH * DV
    cell = _RectCell(NH, DK, DV).to(dev)
    skip = torch.nn.Parameter(1.0 + 0.1 * torch.randn(Hv, device=dev))
    qk0 = 0.5 * torch.randn(B, S, 2 * Hqk, device=dev)
    v0 = torch.randn(B, S, Hv, device=dev)
    x0 = torch.randn(B, S, Hv, device=dev)
    dy = torch.randn(B, S, Hv, device=dev)
    params = dict(ifgate_w=cell.ifgate.weight, ifgate_b=cell.ifgate.bias, ln_w=cell.outnorm.weight,
                  ln_b=cell.outnorm.bias, skip=skip)

    def run(one_launch):
        for p_ in params.values():
            p_.grad = None
        qk, v, x = (t.clone().requires_grad_(True) for t in (qk0, v0, x0))
        q, k = torch.chunk(qk, 2, -1)
        with torch.autocast("cuda", dtype=torch.float16):  # fp16 kernels (kernel_dtype="input") under fp16 autocast, fp16 y
            y = pkg.mlstm_cell_b200(cell, q, k, v, reverse=reverse, skip=skip, x_skip=x, qk=qk, one_launch=one_launch,
                                    kernel_dtype="input")
        assert y.shape == (B, S, Hv) and y.dtype == torch.float16
        n_fw = pkg.last_launch_count()
        y.float().backward(dy)
        out = dict(y=y.detach(), dqk=qk.grad, dv=v.grad, dx=x.grad)
        out.update({n: p_.grad.clone() for n, p_ in params.items()})
        return out, n_fw

    leaves = [t.double().requires_grad_(True) for t in (qk0, v0, x0)]
    pd = {n: p_.detach().double().requires_grad_(True) for n, p_ in params.items()}
    yr = _reference_cell(NH, cell.gate_soft_cap, pd["ifgate_w"], pd["ifgate_b"], 1.0 + pd["ln_w"], pd["ln_b"],
                         cell.outnorm.eps, *leaves, pd["skip"], reverse)
    yr.backward(dy.double())
    want = dict(y=yr, dqk=leaves[0].grad, dv=leaves[1].grad, dx=leaves[2].grad)
    want.update({n: t.grad for n, t in pd.items()})

    got = {mode: run(mode) for mode in ("always", "never", "auto")}
    assert got["always"][1] == 1  # the fused forward is one launch
    # same h, same backward kernels: the two compositions differ by the rounding of y only
    agree = {n: rel(got["always"][0][n], got["never"][0][n]) for n in want}
    assert all(e < 5e-3 for e in agree.values()), agree
    errs = {(mode, n): rel(out[n], w) for mode, (out, _) in got.items() for n, w in want.items()}
    assert all(e < 2e-2 for e in errs.values()), errs
