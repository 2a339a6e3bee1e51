"""torch.compile / torch.export over the ``mlstm_b200`` custom ops (xlstm_yolo_clean_b200/ops.py) on the B200.

A compiled call runs the same kernels on the same inputs as the eager one, so where Inductor only moves tensors between
the ops (the mLSTM calls, the cell output, RMSNorm) the results are compared bit for bit.  The stand-in layer adds
Linear / conv / SiLU around the ops, which Inductor fuses in its own order: it is compared bit for bit with the
``aot_eager`` backend (same graph, eager kernels) and with a tolerance under Inductor."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
HEAD_DIMS = [(32, 32), (64, 64), (128, 128), (32, 64), (64, 128)]


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as G

    G.build()
    import xlstm_yolo_clean_b200 as p

    return p


@pytest.fixture(autouse=True)
def _fresh_dynamo():
    torch._dynamo.reset()
    yield
    torch._dynamo.reset()


def _inputs(B, NH, S, DK, DV, dtype, seed=0, grad=True):
    g = torch.Generator(device="cpu").manual_seed(seed)
    mk = lambda *s, scale=1.0: (torch.randn(*s, generator=g) * scale).to(DEV, dtype).requires_grad_(grad)  # noqa: E731
    q, k = mk(B, NH, S, DK), mk(B, NH, S, DK)
    v = mk(B, NH, S, DV)
    i = mk(B, NH, S, scale=0.5)
    f = (torch.randn(B, NH, S, generator=g) + 3.0).to(DEV, dtype).requires_grad_(grad)
    return q, k, v, i, f


def _grads(ts):
    return [None if t.grad is None else t.grad.clone() for t in ts]


def _run(fn, ts, douts):
    for t in ts:
        t.grad = None
    outs = fn(*ts)
    outs = outs if isinstance(outs, tuple) else (outs,)
    flat = [o for o in outs if o is not None]
    torch.autograd.backward(flat, douts[:len(flat)])
    return [o.detach().clone() for o in flat], _grads(ts)


def _assert_same(a, b):
    for x, y in zip(a, b):
        if x is None or y is None:
            assert x is None and y is None
            continue
        assert x.dtype == y.dtype and x.shape == y.shape
        assert torch.equal(x, y), float((x.float() - y.float()).abs().max())


# ---------------------------------------------------------------------------------------------------------------------
def test_opcheck_every_op(pkg):
    ops = torch.ops.mlstm_b200
    B, NH, S, D = 2, 2, 128, 64
    q, k, v, i, f = _inputs(B, NH, S, D, D, torch.bfloat16)
    fw_args = (q, k, v, i, f, None, None, None, None, None, True, 64, 1e-6, 0, True, False, False, 0.0, None)
    torch.library.opcheck(ops.chunkwise_fw, fw_args)
    h, nm, _, _, _, cs = (t.detach() for t in ops.chunkwise_fw(*fw_args))
    qd, kd, vd, idd, fd = (t.detach() for t in (q, k, v, i, f))
    torch.library.opcheck(ops.chunkwise_bw, (qd, kd, vd, idd, fd, nm[0], nm[1], torch.randn_like(h), None, None, None, None,
                                             cs, None, None, 64, 1e-6, 0, False, False, False, 0.0, torch.float16))
    H = NH * D
    qk = torch.randn(B, S, 2 * H, device=DEV, dtype=torch.float16, requires_grad=True)
    vl = torch.randn(B, S, H, device=DEV, dtype=torch.float16, requires_grad=True)
    gates = torch.randn(B, S, 2 * NH, device=DEV, dtype=torch.float16, requires_grad=True)
    lay = (qk, vl, gates, NH, torch.bfloat16, 64, 1e-6, 0, True, True, False, 15.0, torch.float16)
    torch.library.opcheck(ops.layer_fw, lay)
    hl, nml, csl = (t.detach() for t in ops.layer_fw(*lay))
    torch.library.opcheck(ops.layer_bw, (qk.detach(), vl.detach(), gates.detach(), nml, torch.randn_like(hl), csl, NH,
                                         torch.bfloat16, 64, 1e-6, 0, True, False, 15.0, torch.float16))
    w = torch.randn(H, device=DEV, requires_grad=True)
    b = torch.randn(H, device=DEV, requires_grad=True)
    sk = torch.randn(H, device=DEV, requires_grad=True)
    xs = torch.randn(B, S, H, device=DEV, dtype=torch.float16, requires_grad=True)
    torch.library.opcheck(ops.chunkwise_fw_epilogue, (qk, vl, gates, xs, w, b, sk, NH, torch.bfloat16, 64, 1e-6, 0, True, False,
                                                      False, 15.0, 1e-6, torch.float16, torch.float16))
    hc = torch.randn(B, NH, S, D, device=DEV, dtype=torch.bfloat16, requires_grad=True)
    torch.library.opcheck(ops.cellout_fw, (hc, w, b, sk, xs, 1e-6, torch.float16))
    torch.library.opcheck(ops.cellout_bw, (hc.detach(), xs.detach(), w.detach(), sk.detach(),
                                           torch.randn(B, S, H, device=DEV, dtype=torch.float16), 1e-6, torch.float16, True))
    x = torch.randn(4, 50, 256, device=DEV, dtype=torch.float16).reshape(-1, 256).requires_grad_(True)
    wn = torch.randn(256, device=DEV, requires_grad=True)
    torch.library.opcheck(ops.rmsnorm_fw, (x, wn, 1e-6, torch.float16))
    rstd = ops.rmsnorm_fw(x, wn, 1e-6, torch.float16)[1].detach()
    torch.library.opcheck(ops.rmsnorm_bw, (x.detach(), wn.detach(), rstd, torch.randn_like(x).detach(), 1e-6, torch.float16))
    torch.library.opcheck(ops.convert16, (torch.randn(3, 70, 8, device=DEV, dtype=torch.float16).requires_grad_(True),
                                          torch.bfloat16))
    torch.library.opcheck(ops.recurrent_sequence, (qd[:, :, :16], kd[:, :, :16], vd[:, :, :16], idd[:, :, :16],
                                                   fd[:, :, :16], None, None, None, True, 1e-6, False))


# ---------------------------------------------------------------------------------------------------------------------
def _dropin(pkg, siging=False, **kw):
    fn = pkg.mlstm_siging_chunkwise__b200 if siging else pkg.mlstm_chunkwise__b200

    def f(q, k, v, i, f_, *states):
        st = dict(zip(("c_initial", "n_initial", "m_initial"), states))
        if siging:
            st.pop("m_initial", None)
        out = fn(q, k, v, i, f_, chunk_size=64, eps=1e-6, **st, **kw)
        if kw.get("return_last_states"):
            h, last = out
            return (h, *last)
        return out

    return f


@pytest.mark.parametrize("siging", [False, True])
def test_no_graph_breaks_dropin(pkg, siging):
    q, k, v, i, f = _inputs(2, 4, 256, 64, 64, torch.bfloat16)
    ex = torch._dynamo.explain(_dropin(pkg, siging))(q, k, v, i, f)
    assert ex.graph_break_count == 0 and ex.graph_count == 1, ex.break_reasons


@pytest.mark.parametrize("DK,DV", HEAD_DIMS)
@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("states", [False, True])
def test_fullgraph_dropin_matches_eager(pkg, DK, DV, reverse, states):
    B, NH, S = 2, 3, 192
    ts = list(_inputs(B, NH, S, DK, DV, torch.bfloat16, seed=DK + DV))
    kw = dict(reverse=reverse)
    if states:
        g = torch.Generator(device="cpu").manual_seed(3)
        ts += [(torch.randn(B, NH, DK, DV, generator=g) * 0.1).to(DEV).requires_grad_(True),
               (torch.randn(B, NH, DK, generator=g) * 0.1).to(DEV).requires_grad_(True),
               torch.randn(B, NH, 1, generator=g).to(DEV).requires_grad_(True)]
        kw["return_last_states"] = True
    fn = _dropin(pkg, **kw)
    douts = [torch.randn(B, NH, S, DV, device=DEV, dtype=torch.bfloat16)]
    if states:
        douts += [torch.randn(B, NH, DK, DV, device=DEV, dtype=torch.bfloat16), torch.zeros(B, NH, DK, device=DEV,
                  dtype=torch.bfloat16), torch.zeros(B, NH, 1, device=DEV, dtype=torch.bfloat16)]
    o_e, g_e = _run(fn, ts, douts)
    n_eager = pkg.last_launch_count()
    o_c, g_c = _run(torch.compile(fn, fullgraph=True), ts, douts)
    assert pkg.last_launch_count() == n_eager
    _assert_same(o_e, o_c)
    _assert_same(g_e, g_c)


@pytest.mark.parametrize("siging", [False, True])
def test_fullgraph_fp16_autocast_bf16_kernel(pkg, siging):
    """custom_fwd(cast_inputs=bf16) under fp16 autocast: the compiled call rounds the fp16 inputs to bf16 inside the op
    and the backward writes fp16 gradients straight from the kernel, as the eager call does."""
    ts = _inputs(2, 4, 320, 64, 64, torch.float16, seed=11)
    fn = _dropin(pkg, siging)

    def under_amp(*a):
        with torch.autocast("cuda", dtype=torch.float16):
            return fn(*a)

    dh = [torch.randn(2, 4, 320, 64, device=DEV, dtype=torch.bfloat16)]
    o_e, g_e = _run(under_amp, ts, dh)
    o_c, g_c = _run(torch.compile(under_amp, fullgraph=True), ts, dh)
    assert o_e[0].dtype == torch.bfloat16 and all(g.dtype == torch.float16 for g in g_e)
    _assert_same(o_e, o_c)
    _assert_same(g_e, g_c)


def test_dynamic_batch_does_not_recompile(pkg):
    from torch._dynamo.testing import CompileCounterWithBackend

    cnt = CompileCounterWithBackend("inductor")
    fn = torch.compile(_dropin(pkg), backend=cnt, fullgraph=True)
    for B in (2, 3, 5):
        ts = _inputs(B, 4, 128, 64, 64, torch.bfloat16, seed=B)
        for t in ts:
            torch._dynamo.mark_dynamic(t, 0)
        o_c, g_c = _run(fn, ts, [torch.ones(B, 4, 128, 64, device=DEV, dtype=torch.bfloat16)])
        o_e, g_e = _run(_dropin(pkg), ts, [torch.ones(B, 4, 128, 64, device=DEV, dtype=torch.bfloat16)])
        _assert_same(o_e, o_c)
        _assert_same(g_e, g_c)
    assert cnt.frame_count == 1, cnt.frame_count


def test_reduce_overhead_replays_match_eager(pkg):
    fn = _dropin(pkg)
    cfn = torch.compile(fn, mode="reduce-overhead", fullgraph=True)
    for seed in range(5):  # the first calls record, the later ones replay; three input sets are checked after warm-up
        ts = _inputs(2, 4, 256, 64, 64, torch.bfloat16, seed=100 + seed % 3)
        dh = [torch.randn(2, 4, 256, 64, device=DEV, dtype=torch.bfloat16)]
        o_c, g_c = _run(cfn, ts, dh)
        o_e, g_e = _run(fn, ts, dh)
        _assert_same(o_e, o_c)
        _assert_same(g_e, g_c)


def test_public_fw_bw_and_convert16_compile(pkg):
    q, k, v, i, f = (t.detach() for t in _inputs(2, 4, 128, 64, 64, torch.bfloat16, seed=5))
    dh = torch.randn(2, 4, 128, 64, device=DEV, dtype=torch.bfloat16)

    def fwbw(q, k, v, i, f, dh):
        h, n, m, _, cs = pkg.mlstm_chunkwise_fw(q, k, v, i, f)
        return (h, *pkg.mlstm_chunkwise_bw(q, k, v, i, f, n, m, dh, c_states=cs)[:5], pkg.convert16(h, torch.float16))

    e = fwbw(q, k, v, i, f, dh)
    c = torch.compile(fwbw, fullgraph=True)(q, k, v, i, f, dh)
    _assert_same(e, c)


def test_recurrent_sequence_compiles(pkg):
    q, k, v, i, f = (t.detach() for t in _inputs(2, 4, 24, 64, 64, torch.bfloat16, seed=9))

    def rec(q, k, v, i, f):
        h, (c, n, m) = pkg.mlstm_recurrent_sequence__b200(q, k, v, i, f, return_last_states=True)
        h1, (c1, n1, m1) = pkg.mlstm_recurrent_step__b200(q[:, :, 0], k[:, :, 0], v[:, :, 0], i[:, :, :1], f[:, :, :1], c, n, m)
        return h, c, n, m, h1, c1, n1, m1

    ex = torch._dynamo.explain(rec)(q, k, v, i, f)
    assert ex.graph_break_count == 0, ex.break_reasons
    _assert_same(rec(q, k, v, i, f), torch.compile(rec, fullgraph=True)(q, k, v, i, f))


# ---------------------------------------------------------------------------------------------------------------------
# a ViLLayer stand-in (modelled on tests/test_cell_gpu.py's _Layer) with optional rectangular heads
class _Norm(torch.nn.Module):
    def __init__(self, H):
        super().__init__()
        self.weight = torch.nn.Parameter(0.1 * torch.randn(H))
        self.bias = torch.nn.Parameter(0.1 * torch.randn(H))
        self.eps = 1e-6

    @property
    def weight_proxy(self):
        return 1.0 + self.weight


class _Cell(torch.nn.Module):
    def __init__(self, H, Hqk, NH):
        super().__init__()
        self.dim, self.num_heads, self.gate_soft_cap = H, NH, 15.0
        self.use_autocast, self.autocast_dtype = True, torch.float16
        self.ifgate = torch.nn.Linear(2 * Hqk + H, 2 * NH)
        self.outnorm = _Norm(H)
        with torch.no_grad():
            self.ifgate.bias[:NH] = -2.0
            self.ifgate.bias[NH:] = torch.linspace(3.0, 6.0, NH)


class _Dir:
    def __init__(self, name):
        self.name = name


class _Layer(torch.nn.Module):
    def __init__(self, dim, NH, reverse, qk_factor=1.0):
        super().__init__()
        inner = 2 * dim
        Hqk = int(inner * qk_factor)
        self.direction = _Dir("ROWWISE_FROM_BOT_RIGHT" if reverse else "ROWWISE_FROM_TOP_LEFT")
        self.proj_up = torch.nn.Linear(dim, 2 * inner)
        self.conv = torch.nn.Conv2d(inner, inner, 3, padding=1, groups=inner)
        self.qk_proj = torch.nn.Linear(inner, 2 * Hqk)
        self.v_proj = torch.nn.Linear(inner, inner)
        self.mlstm_cell = _Cell(inner, Hqk, NH)
        self.learnable_skip = torch.nn.Parameter(1.0 + 0.1 * torch.randn(inner))
        self.proj_down = torch.nn.Linear(inner, dim)
        self.norm = torch.nn.RMSNorm(dim, eps=1e-6)
        with torch.no_grad():
            self.norm.weight.add_(0.1 * torch.randn(dim))


class _Block(torch.nn.Module):
    """x + mlstm_branch(RMSNorm(x)) under fp16 autocast, like ViLLayer.forward in the ultralytics trainer."""

    def __init__(self, pkg, layer, one_launch, amp=True):
        super().__init__()
        self.layer, self.one_launch, self.amp, self.pkg = layer, one_launch, amp, pkg

    def forward(self, x):
        with torch.autocast("cuda", dtype=torch.float16, enabled=self.amp):
            y = self.pkg.rms_norm_b200(x, self.layer.norm.weight, 1e-6)
            return x + self.pkg.mlstm_branch_b200(self.layer, y, one_launch=self.one_launch)


def _block_run(block, x, dout, fn=None):
    block.zero_grad()
    xi = x.clone().requires_grad_(True)
    out = (block if fn is None else fn)(xi)
    out.backward(dout)
    grads = {n: p.grad.clone() for n, p in block.named_parameters() if p.grad is not None}
    return out.detach().float(), xi.grad.clone(), grads


def _make_block(pkg, reverse, one_launch, qk_factor=1.0, dim=256, NH=8, seed=5):  # base256: 8 heads of 64
    torch.manual_seed(seed)
    return _Block(pkg, _Layer(dim, NH, reverse, qk_factor).to(DEV), one_launch)


@pytest.mark.parametrize("one_launch", ["auto", "always"])
def test_no_graph_breaks_layer(pkg, one_launch):
    block = _make_block(pkg, True, one_launch)
    x = torch.randn(2, 256, 256, device=DEV, requires_grad=True)
    ex = torch._dynamo.explain(block)(x)
    assert ex.graph_break_count == 0 and ex.graph_count == 1, ex.break_reasons


@pytest.mark.parametrize("one_launch", ["auto", "always"])
@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("qk_factor,S", [(1.0, 256), (0.5, 256), (1.0, 100)])
def test_layer_aot_eager_bit_identical_inductor_close(pkg, one_launch, reverse, qk_factor, S):
    block = _make_block(pkg, reverse, one_launch, qk_factor)
    x = torch.randn(2, S, 256, device=DEV)
    dout = torch.randn(2, S, 256, device=DEV)
    o_e, dx_e, g_e = _block_run(block, x, dout)
    o_a, dx_a, g_a = _block_run(block, x, dout, torch.compile(block, backend="aot_eager", fullgraph=True))
    assert torch.equal(o_e, o_a) and torch.equal(dx_e, dx_a)
    assert set(g_e) == set(g_a) and all(torch.equal(g_e[n], g_a[n]) for n in g_e)
    torch._dynamo.reset()
    o_i, dx_i, g_i = _block_run(block, x, dout, torch.compile(block, fullgraph=True))

    def rel(a, b):
        return float((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))

    # Inductor's own fusion of the dense layers around the ops re-rounds fp16 intermediates differently
    assert rel(o_i, o_e) < 1e-2 and rel(dx_i, dx_e) < 3e-2
    assert all(rel(g_i[n], g_e[n]) < 5e-2 for n in g_e), {n: rel(g_i[n], g_e[n]) for n in g_e}


def test_export_standin_forward(pkg):
    block = _make_block(pkg, True, "always")
    x = torch.randn(2, 256, 256, device=DEV)
    with torch.no_grad():
        ep = torch.export.export(block, (x,))
        want = block(x)
        got = ep.module()(x)
    assert torch.equal(want, got)


@pytest.mark.parametrize("C", [192, 256])
def test_rmsnorm_and_cell_out_fullgraph(pkg, C):
    x = torch.randn(3, 77, C, device=DEV, dtype=torch.float16, requires_grad=True)
    w = (1.0 + 0.2 * torch.randn(C, device=DEV)).requires_grad_(True)
    h = torch.randn(3, 4, 77, 64, device=DEV, dtype=torch.bfloat16, requires_grad=True)
    hw, hb, hs = (torch.randn(256, device=DEV, requires_grad=True) for _ in range(3))
    xs = torch.randn(3, 77, 256, device=DEV, dtype=torch.float16, requires_grad=True)

    def f(x, w, h, hw, hb, hs, xs):
        with torch.autocast("cuda", dtype=torch.float16):
            return pkg.rms_norm_b200(x, w, 1e-6), pkg.cell_out(h, hw, hb, hs, xs, eps=1e-6)

    ts = [x, w, h, hw, hb, hs, xs]
    douts = [torch.randn(3, 77, C, device=DEV, dtype=torch.float16), torch.randn(3, 77, 256, device=DEV, dtype=torch.float16)]
    ex = torch._dynamo.explain(f)(*ts)
    assert ex.graph_break_count == 0, ex.break_reasons
    o_e, g_e = _run(f, ts, douts)
    o_c, g_c = _run(torch.compile(f, fullgraph=True), ts, douts)
    _assert_same(o_e, o_c)
    _assert_same(g_e, g_c)


@pytest.mark.parametrize("backend", ["inductor", "aot_eager"])
def test_cell_out_misaligned_skip_input(pkg, backend):
    """A contiguous skip input 2 bytes past an aligned address (the cell-output kernels need 8): eager and compiled calls
    both read an aligned copy and agree bit for bit."""
    n = 3 * 77 * 256
    xs = torch.randn(n + 1, device=DEV, dtype=torch.float16)[1:].view(3, 77, 256).requires_grad_(True)
    assert xs.is_leaf and xs.data_ptr() % 8
    h = torch.randn(3, 4, 77, 64, device=DEV, dtype=torch.bfloat16, requires_grad=True)
    hw, hb, hs = (torch.randn(256, device=DEV, requires_grad=True) for _ in range(3))

    def f(h, hw, hb, hs, xs):
        with torch.autocast("cuda", dtype=torch.float16):
            return pkg.cell_out(h, hw, hb, hs, xs, eps=1e-6)

    ts = [h, hw, hb, hs, xs]
    douts = [torch.randn(3, 77, 256, device=DEV, dtype=torch.float16)]
    o_e, g_e = _run(f, ts, douts)
    o_c, g_c = _run(torch.compile(f, backend=backend, fullgraph=True), ts, douts)
    _assert_same(o_e, o_c)
    _assert_same(g_e, g_c)
