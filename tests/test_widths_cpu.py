"""Which ViL widths get the fused layer path (vil.cellout_supported / vil.rmsnorm_supported / vil.patch_layers), without a
GPU: the documented support matrix at and just outside each boundary, and patch_layers' count of rebound layers on
stand-ins of every width the GPU tests run."""
import warnings

import pytest
import torch


@pytest.fixture(scope="module")
def vil():
    import xlstm_yolo_clean_b200.vil as v

    return v


@pytest.mark.parametrize("D", [32, 64, 128])
def test_cellout_matrix(vil, D):
    for NH in range(1, 2048 // D + 1):  # every head count up to NH * D = 2048, multiples of 128 or not
        assert vil.cellout_supported(NH, D), (NH, D)
    assert not vil.cellout_supported(2048 // D + 1, D)
    assert not vil.cellout_supported(0, D)


@pytest.mark.parametrize("D", [16, 48, 96, 256])
def test_cellout_other_head_dims(vil, D):
    assert not any(vil.cellout_supported(NH, D) for NH in (1, 2, 3, 4, 8))


def test_rmsnorm_matrix(vil):
    covered = [C for C in range(0, 4097) if vil.rmsnorm_supported(C)]
    assert covered == list(range(64, 2049, 32))
    for C in (32, 63, 65, 100, 2047, 2049, 2080):
        assert not vil.rmsnorm_supported(C)


class _Cell(torch.nn.Module):
    def __init__(self, H, NH):
        super().__init__()
        self.dim, self.num_heads = H, NH


class _StandIn(torch.nn.Module):
    """Attribute-shaped ViLLayer (vision_lstm2.py:218-290) of width ``dim``: NH = 2 dim / qkv_block_size heads of
    head dim qkv_block_size.  Only what patch_layers looks at; nothing runs."""

    def __init__(self, dim, qkv_block_size):
        super().__init__()
        inner = 2 * dim
        self.proj_up = self.qk_proj = self.v_proj = self.proj_down = torch.nn.Identity()
        self.mlstm_cell = _Cell(inner, inner // qkv_block_size)
        self.learnable_skip = torch.nn.Parameter(torch.ones(inner))
        self.norm, self.ffn_norm = torch.nn.RMSNorm(dim, eps=1e-6), torch.nn.RMSNorm(dim, eps=1e-6)


# (dim, qkv_block_size): the GPU tests' widths, the shipped ones and two more
WIDTHS = [(96, 32), (160, 64), (320, 128), (448, 64), (192, 32), (256, 64), (384, 128), (128, 32), (640, 64),
          (768, 128), (1024, 128), (224, 32), (288, 64)]


def test_patch_layers_rebinds_every_width(vil):
    model = torch.nn.Sequential(*[_StandIn(d, q) for d, q in WIDTHS])
    with warnings.catch_warnings():
        warnings.simplefilter("error")  # nothing is skipped: no warning
        assert vil.patch_layers(model) == len(WIDTHS)
    for layer in model:
        assert "mlstm_branch" in layer.__dict__
        assert "forward" in layer.norm.__dict__ and "forward" in layer.ffn_norm.__dict__


def test_patch_layers_names_what_it_skips(vil):
    # H = 2304 > 2048; head dim 48; RMSNorm of width 100 (not a multiple of 32) on an otherwise covered layer
    big, odd, ok = _StandIn(1152, 128), _StandIn(192, 48), _StandIn(100, 40)
    ok.mlstm_cell = _Cell(256, 4)
    model = torch.nn.ModuleDict(dict(big=big, odd=odd, ok=ok))
    with pytest.warns(UserWarning, match=r"2 ViL layer\(s\) left unpatched.*big \(NH=18, D=128\), odd \(NH=8, D=48\)"):
        assert vil.patch_layers(model) == 1
    assert "mlstm_branch" not in big.__dict__ and "forward" not in big.norm.__dict__
    assert "mlstm_branch" not in odd.__dict__
    assert "mlstm_branch" in ok.__dict__ and "forward" not in ok.norm.__dict__
