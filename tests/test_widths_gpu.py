"""The fused ViL layer path at every model width (tests/test_widths_cpu.py has the support matrix): the cell-output
kernels at row widths H = NH * D that are not multiples of 128 (a tail warp covers H mod 128 channels), the RMSNorm at
every C that is a multiple of 32 from 64 to 2048, the one-launch fused cell and whole patched ViLLayer stand-ins at
widths other than the three shipped ones.

Checkers: float64 torch composites (F.group_norm + relayout + skip; x * rsqrt(mean(x^2) + eps) * w), torch.rms_norm
itself, the two-launch cell, and the unpatched layer.  Tolerances: 1e-5 relative for fp32 tensors, 2e-2 where a
16-bit rounding is part of the function; the layer comparisons use those of tests/test_cell_gpu.py."""
import copy

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
DTYPES = (torch.bfloat16, torch.float16, torch.float32)


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as G

    G.build()
    import xlstm_yolo_clean_b200 as p

    return p


def rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def tol(dtype):
    return 1e-5 if dtype == torch.float32 else 2e-2


# ---------------------------------------------------------------------------------------------------------------------
# cell output
def ref_cell_out(h, weight, bias, skip, x, eps):
    """MultiHeadLayerNorm (vision_lstm2.py:928-944) + relayout + skip (vision_lstm2.py:306), in h's dtype (float64)."""
    B, NH, S, D = h.shape
    y = F.group_norm(h.transpose(1, 2).reshape(B * S, NH * D), NH, weight, bias, eps).view(B, S, NH * D)
    return y + skip * x if x is not None else y


# tail rows (H mod 128 = 32, 64 or 96) and, as controls, two widths the tail-free kernels run
CELL_SHAPES = [(3, 32), (5, 32), (3, 64), (5, 64), (7, 64), (63, 32), (5, 128), (16, 128)]
CELL_IDS = [f"H{nh * d}_{nh}x{d}" for nh, d in CELL_SHAPES]


def _cell_case(pkg, h, x_dtype, with_params, with_skip, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    B, NH, S, D = h.shape
    H = NH * D
    h = h.requires_grad_(True)
    w = (1.0 + 0.2 * torch.randn(H, generator=g)).to(DEV).requires_grad_(True) if with_params else None
    b = (0.1 * torch.randn(H, generator=g)).to(DEV).requires_grad_(True) if with_params else None
    sk = (1.0 + 0.1 * torch.randn(H, generator=g)).to(DEV).requires_grad_(True) if with_skip else None
    x = torch.randn(B, S, H, generator=g).to(x_dtype).to(DEV).requires_grad_(True) if with_skip else None
    dy = torch.randn(B, S, H, generator=g).to(x_dtype).to(DEV)
    y = pkg.cell_out(h, w, b, sk, x, eps=1e-6, out_dtype=x_dtype)
    assert y.shape == (B, S, H) and y.dtype == x_dtype
    y.backward(dy)
    leaves = {k: t for k, t in dict(h=h, x=x, w=w, b=b, sk=sk).items() if t is not None}
    ref = {k: t.detach().double().requires_grad_(True) for k, t in leaves.items()}
    yr = ref_cell_out(ref["h"], ref.get("w"), ref.get("b"), ref.get("sk"), ref.get("x"), 1e-6)
    yr.backward(dy.double())
    assert rel(y, yr) < tol(x_dtype), ("y", rel(y, yr))
    for k, t in leaves.items():
        want = tol(h.dtype) if k == "h" else tol(x_dtype) if k == "x" else 1e-5
        assert rel(t.grad, ref[k].grad) < want, (k, rel(t.grad, ref[k].grad), want)


@pytest.mark.parametrize("NH,D", CELL_SHAPES, ids=CELL_IDS)
@pytest.mark.parametrize("h_dtype", DTYPES)
@pytest.mark.parametrize("x_dtype", DTYPES)
def test_cell_out_any_width(pkg, NH, D, h_dtype, x_dtype):
    """Every (h, y) dtype pair the kernels accept, weight + bias + skip, against float64."""
    B, S = 2, 97
    h = (torch.randn(B, NH, S, D, generator=torch.Generator().manual_seed(NH * D)) * 1.7 + 0.3).to(h_dtype).to(DEV)
    _cell_case(pkg, h, x_dtype, True, True, NH + D)


@pytest.mark.parametrize("NH,D", CELL_SHAPES, ids=CELL_IDS)
@pytest.mark.parametrize("layout", ["s_slice", "layer_view"])
def test_cell_out_any_width_strided_h_without_params(pkg, NH, D, layout):
    """h as a slice of a longer (B, NH, S', D) buffer (the padded call) or as the (B, NH, S, D) view of a (B, S, NH D)
    tensor (the layer layout), with no weight / bias / skip, and with weight + bias but no skip."""
    B, S = 2, 100
    g = torch.Generator().manual_seed(7 * NH + D)
    if layout == "s_slice":
        h = torch.randn(B, NH, S + 28, D, generator=g).to(torch.bfloat16).to(DEV)[:, :, 28:]
    else:
        h = torch.randn(B, S, NH * D, generator=g).to(torch.bfloat16).to(DEV).view(B, S, NH, D).transpose(1, 2)
    assert not h.is_contiguous()
    _cell_case(pkg, h.detach(), torch.float16, False, False, NH)
    _cell_case(pkg, h.detach(), torch.float32, True, False, NH + 1)


def test_cell_out_tail_width_is_deterministic(pkg):
    B, NH, S, D = 4, 5, 1600, 32
    h = torch.randn(B, NH, S, D, device=DEV).to(torch.bfloat16).requires_grad_(True)
    x = torch.randn(B, S, NH * D, device=DEV).to(torch.float16)
    w, sk = (torch.randn(NH * D, device=DEV).requires_grad_(True) for _ in range(2))
    dy = torch.randn(B, S, NH * D, device=DEV).to(torch.float16)
    outs = []
    for _ in range(2):
        h.grad = w.grad = sk.grad = None
        pkg.cell_out(h, w, None, sk, x, out_dtype=torch.float16).backward(dy)
        outs.append((h.grad.clone(), w.grad.clone(), sk.grad.clone()))
    for a, b in zip(*outs):
        assert torch.equal(a, b)


def test_cell_out_rejects_rows_wider_than_2048(pkg):
    with pytest.raises(RuntimeError, match="2048"):
        pkg.cell_out(torch.randn(1, 17, 8, 128, device=DEV))


# ---------------------------------------------------------------------------------------------------------------------
# RMSNorm
RMS_WIDTHS = [64, 96, 128, 160, 320, 448, 640, 768, 1024, 2048, 544, 1056, 2016]


@pytest.mark.parametrize("C", RMS_WIDTHS)
@pytest.mark.parametrize("x_dtype,y_dtype", [(torch.float16, torch.float16), (torch.float32, torch.float16),
                                             (torch.float32, torch.float32), (torch.bfloat16, torch.float32)])
def test_rms_norm_any_width(pkg, C, x_dtype, y_dtype):
    torch.manual_seed(C)
    x = (torch.randn(5, 77, C, device=DEV) * 1.3 + 0.2).to(x_dtype).requires_grad_(True)
    w = (1.0 + 0.2 * torch.randn(C, device=DEV)).requires_grad_(True)
    dy = torch.randn(5, 77, C, device=DEV).to(y_dtype)
    y = pkg.rms_norm_b200(x, w, 1e-6, out_dtype=y_dtype)
    assert y.shape == x.shape and y.dtype == y_dtype
    y.backward(dy)
    want = torch.rms_norm(x.detach(), (C,), w.detach(), 1e-6)
    tol_y = {torch.float32: 2e-6, torch.float16: 1e-3, torch.bfloat16: 8e-3}
    assert rel(y, want) < max(tol_y[y_dtype], tol_y[x_dtype]), rel(y, want)
    x64, w64 = x.detach().double().requires_grad_(True), w.detach().double().requires_grad_(True)
    (x64 * torch.rsqrt(x64.pow(2).mean(-1, keepdim=True) + 1e-6) * w64).backward(dy.double())
    assert rel(x.grad, x64.grad) < max(tol_y[x_dtype], 2e-3), rel(x.grad, x64.grad)
    assert rel(w.grad, w64.grad) < max(tol_y[x_dtype], 2e-3), rel(w.grad, w64.grad)
    dw = w.grad.clone()
    w.grad = None
    pkg.rms_norm_b200(x, w, 1e-6, out_dtype=y_dtype).backward(dy)
    assert torch.equal(w.grad, dw)  # two-stage reduction in a fixed order


@pytest.mark.parametrize("C", [96, 160, 640, 2048])
def test_rms_norm_any_width_autocast_rounding(pkg, C):
    """Under fp16 autocast (fp16 input, fp32 weight) the output is rounded once to the input dtype, as torch's
    composite does: at most one fp16 ulp apart (summation order of mean(x^2)), on a small fraction of elements."""
    torch.manual_seed(C + 1)
    norm = torch.nn.RMSNorm(C, eps=1e-6).to(DEV)
    with torch.no_grad():
        norm.weight.add_(0.3 * torch.randn(C, device=DEV))
    x = torch.randn(4, 400, C, device=DEV).half()
    with torch.autocast("cuda", dtype=torch.float16):
        a = norm(x).to(torch.float16)
        b = pkg.rms_norm_b200(x, norm.weight, norm.eps)
    assert b.dtype == torch.float16
    diff = (a.float() - b.float()).abs()
    assert float((diff / a.float().abs().clamp_min(1e-3)).max()) <= 2.0 ** -9
    assert float((diff > 0).float().mean()) < 0.02


def test_rms_norm_rejects_uncovered_widths(pkg):
    for C in (32, 100, 2080):
        with pytest.raises(RuntimeError, match="not covered"):
            pkg.rms_norm_b200(torch.randn(4, C, device=DEV), torch.ones(C, device=DEV))


# ---------------------------------------------------------------------------------------------------------------------
# stand-ins (tests/test_cell_gpu.py has the same ones for the shipped widths)
class _Norm(torch.nn.Module):
    def __init__(self, H):
        super().__init__()
        self.weight = torch.nn.Parameter(0.1 * torch.randn(H))
        self.bias = torch.nn.Parameter(0.1 * torch.randn(H))
        self.eps = 1e-6

    @property
    def weight_proxy(self):
        return 1.0 + self.weight


class _Conv(torch.nn.Conv2d):
    seqlens = None


class _Cell(torch.nn.Module):
    def __init__(self, H, NH):
        super().__init__()
        self.dim, self.num_heads, self.gate_soft_cap = H, NH, 15.0
        self.use_autocast, self.autocast_dtype = True, torch.float16
        self.ifgate = torch.nn.Linear(3 * H, 2 * NH)
        self.outnorm = _Norm(H)
        with torch.no_grad():
            self.ifgate.bias[:NH] = -2.0
            self.ifgate.bias[NH:] = torch.linspace(3.0, 6.0, NH)


class _Dir:
    def __init__(self, name):
        self.name = name


class _NoDrop(torch.nn.Module):
    drop_prob = 0.0


class _Layer(torch.nn.Module):
    """Attribute-compatible stand-in for a whole ViLLayer (vision_lstm2.py:218-341) of width ``dim`` with
    NH = 2 dim / qkv_block_size heads: norm -> mlstm branch -> residual -> ffn_norm -> ffn -> residual."""

    def __init__(self, dim, qkv_block_size, reverse):
        super().__init__()
        inner = 2 * dim
        NH = inner // qkv_block_size
        self.direction = _Dir("ROWWISE_FROM_BOT_RIGHT" if reverse else "ROWWISE_FROM_TOP_LEFT")
        self.proj_up = torch.nn.Linear(dim, 2 * inner)
        self.conv = _Conv(inner, inner, 3, padding=1, groups=inner)
        self.qk_proj = torch.nn.Linear(inner, 2 * inner)
        self.v_proj = torch.nn.Linear(inner, inner)
        self.mlstm_cell = _Cell(inner, NH)
        self.learnable_skip = torch.nn.Parameter(1.0 + 0.1 * torch.randn(inner))
        self.proj_down = torch.nn.Linear(inner, dim)
        self.norm, self.ffn_norm = torch.nn.RMSNorm(dim, eps=1e-6), torch.nn.RMSNorm(dim, eps=1e-6)
        with torch.no_grad():
            self.norm.weight.add_(0.1 * torch.randn(dim))
            self.ffn_norm.weight.add_(0.1 * torch.randn(dim))
        self.ffn = torch.nn.Sequential(torch.nn.Linear(dim, 2 * dim), torch.nn.GELU(), torch.nn.Linear(2 * dim, dim))
        self.drop_path = _NoDrop()

    def mlstm_branch(self, x):  # the unpatched layer: the reference's composition (replaced by patch_layers)
        return _reference_branch(self, x)

    def forward(self, x):
        x = x + self.mlstm_branch(self.norm(x))
        return x + self.ffn(self.ffn_norm(x))


def _reference_branch(layer, x):
    """ViLLayer.mlstm_branch as the reference composes it (flip, conv, cell with group_norm, skip, flip back), plain
    torch + the causal chunkwise kernel on fp16 heads (MatrixLSTMCell's CUDA cast, vision_lstm2.py:730-745)."""
    import xlstm_yolo_clean_b200 as pkg

    reverse = pkg.vil._is_reverse(layer)
    if reverse:
        x = x.flip(dims=[1])
    B, S, _ = x.shape
    x_qk, x_v = torch.chunk(layer.proj_up(x), 2, dim=-1)
    hh = int(S ** 0.5)
    img = x_qk.reshape(B, hh, hh, -1).permute(0, 3, 1, 2)
    x_act = F.silu(layer.conv(img).permute(0, 2, 3, 1).reshape(B, S, -1))
    q, k = torch.chunk(layer.qk_proj(x_act), 2, dim=-1)
    v = layer.v_proj(x_v)
    cell = layer.mlstm_cell
    NH = cell.num_heads
    pre = cell.ifgate(torch.cat([q, k, v], -1))
    pre = 15.0 * torch.tanh(pre / 15.0)
    i, f = (t.transpose(-1, -2) for t in torch.chunk(pre, 2, -1))
    qh, kh, vh = (t.view(B, S, NH, -1).transpose(1, 2).to(torch.float16) for t in (q, k, v))
    i, f = i.to(torch.float16), f.to(torch.float16)
    pad = (-S) % 64
    if pad:
        qh, kh, vh = (F.pad(t, (0, 0, 0, pad)) for t in (qh, kh, vh))
        i, f = F.pad(i, (0, pad)), F.pad(f, (0, pad))
    h = pkg.mlstm_chunkwise__b200(q=qh, k=kh, v=vh, i=i, f=f, chunk_size=64, eps=1e-6)[:, :, :S].to(x.dtype)
    D = h.shape[-1]
    g = F.group_norm(h.transpose(1, 2).reshape(B * S, NH * D), NH, cell.outnorm.weight_proxy, cell.outnorm.bias, 1e-6)
    out = layer.proj_down(g.view(B, S, NH * D) + layer.learnable_skip * x_act)
    return out.flip(dims=[1]) if reverse else out


# ---------------------------------------------------------------------------------------------------------------------
# one-launch fused cell
@pytest.mark.parametrize("NH,D", [(3, 32), (5, 32), (3, 64), (5, 64), (3, 128), (5, 128)],
                         ids=["H96", "H160", "H192", "H320", "H384", "H640"])
@pytest.mark.parametrize("reverse", [False, True], ids=["causal", "anticausal"])
def test_fused_cell_matches_two_launches(pkg, monkeypatch, NH, D, reverse):
    """_MlstmCellFused (one_launch="always": LayerNorm, relayout and skip in the mLSTM forward's epilogue) against the
    mLSTM kernel followed by the cell-output kernels (one_launch="never"), without gradients and in training."""
    H, B, S = NH * D, 2, 144
    torch.manual_seed(H + reverse)
    cell = _Cell(H, NH).to(DEV)
    skip = torch.nn.Parameter(1.0 + 0.1 * torch.randn(H, device=DEV))
    qk0 = torch.randn(B, S, 2 * H, device=DEV)
    v0, xs0 = torch.randn(B, S, H, device=DEV), torch.randn(B, S, H, device=DEV)
    dy = torch.randn(B, S, H, device=DEV)
    fused_calls = []
    inner = pkg.vil._cell_fused
    monkeypatch.setattr(pkg.vil, "_cell_fused", lambda *a, **k: fused_calls.append(1) or inner(*a, **k))

    def run(one_launch, train):
        params = [*cell.parameters(), skip]
        for p in params:
            p.grad = None
        qk, v, xs = (t.clone().requires_grad_(train) for t in (qk0, v0, xs0))
        with torch.set_grad_enabled(train), torch.autocast("cuda", dtype=torch.float16):
            q, k = torch.chunk(qk, 2, dim=-1)
            y = pkg.mlstm_cell_b200(cell, q, k, v, reverse=reverse, skip=skip, x_skip=xs, qk=qk, one_launch=one_launch)
        if not train:
            return y, []
        y.float().backward(dy)
        return y.detach(), [qk.grad, v.grad, xs.grad] + [p.grad for p in params]

    for train in (False, True):
        n0 = len(fused_calls)
        y1, g1 = run("always", train)
        assert len(fused_calls) == n0 + 1
        y2, g2 = run("never", train)
        assert len(fused_calls) == n0 + 1
        assert y1.dtype == y2.dtype == torch.float16
        assert rel(y1, y2) < 2e-2, (train, rel(y1, y2))
        for a, b in zip(g1, g2):
            assert rel(a, b) < 2e-2, (train, rel(a, b))


# ---------------------------------------------------------------------------------------------------------------------
# whole layers
LAYER_WIDTHS = [(96, 32), (160, 64), (320, 128), (448, 64)]  # (dim, qkv_block_size)


@pytest.mark.parametrize("dim,qkv", LAYER_WIDTHS, ids=[f"dim{d}" for d, _ in LAYER_WIDTHS])
def test_patched_layers_match_unpatched_at_any_width(pkg, dim, qkv):
    """patch_layers on a two-direction stack of ViLLayer stand-ins of width ``dim``: every layer is rebound (branch and
    both RMSNorms), and under fp16 autocast the loss, the input gradient and every parameter gradient match the
    unpatched stack."""
    torch.manual_seed(dim)
    model = torch.nn.Sequential(_Layer(dim, qkv, False), _Layer(dim, qkv, True)).to(DEV)
    for layer in model:
        layer.conv.seqlens = [12, 12]
    x = torch.randn(2, 144, dim, device=DEV)

    def step():
        model.zero_grad()
        xi = x.clone().requires_grad_(True)
        with torch.autocast("cuda", dtype=torch.float16):
            out = model(xi)
            loss = out.float().pow(2).mean()
        loss.backward()
        return float(loss), xi.grad.clone(), {n: p.grad.clone() for n, p in model.named_parameters()}

    loss_ref, dx_ref, g_ref = step()
    assert pkg.patch_layers(model) == 2
    for layer in model:
        assert "mlstm_branch" in layer.__dict__ and "forward" in layer.norm.__dict__ and "forward" in layer.ffn_norm.__dict__
    loss_new, dx_new, g_new = step()
    assert abs(loss_new - loss_ref) < 5e-3 * abs(loss_ref)
    assert rel(dx_new, dx_ref) < 3e-2, rel(dx_new, dx_ref)
    assert set(g_new) == set(g_ref)
    for n in g_ref:
        assert rel(g_new[n], g_ref[n]) < 3e-2, (n, rel(g_new[n], g_ref[n]))


def test_graphed_layer_at_a_tail_width_is_bit_identical_to_eager(pkg):
    """patch_layers(graphs=True) at dim 160 (H = 320 = 2.5 x 128: the cell-output tail warp): the whole layer replays as
    CUDA graphs, bit-identical to the eager patched layer over two optimizer steps."""
    torch.manual_seed(11)
    eager = _Layer(160, 64, True).to(DEV)
    eager.conv.seqlens = [20, 20]
    graphed = copy.deepcopy(eager)
    assert pkg.patch_layers(eager) == 1 and pkg.patch_layers(graphed, graphs=True) == 1
    assert "forward" in graphed.__dict__
    opts = [torch.optim.SGD(m.parameters(), lr=0.05) for m in (eager, graphed)]
    for it in range(2):
        x = torch.randn(4, 400, 160, device=DEV)
        res = []
        for m, opt in zip((eager, graphed), opts):
            xi = x.clone().requires_grad_(True)
            opt.zero_grad()
            with torch.autocast("cuda", dtype=torch.float16):
                y = m(xi)
            loss = (y.float() ** 2).mean()
            loss.backward()
            opt.step()
            res.append((loss.detach(), xi.grad))
        assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1]), it
        for a, b in zip(eager.parameters(), graphed.parameters()):
            assert torch.equal(a, b), it
    assert len(graphed.forward._graphs) == 1
