"""CPU-only checks of the boundary: the C-ABI library loads, exports every symbol the header
declares, and the host shim refuses to run without a GPU (no fallback)."""
import ctypes
import os
import re

import pytest
import torch

import __graft_entry__ as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    G.build()
    import xlstm_yolo_clean_b200 as pkg

    return pkg.load_library()


def _header_functions():
    src = open(os.path.join(ROOT, "include", "mlstm_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mlstm_b200_[a-z_0-9]+)\s*\(", src)))


def test_exports_match_header(lib):
    from xlstm_yolo_clean_b200 import _cabi

    names = _header_functions()
    assert set(names) == set(_cabi.EXPORTS)
    for n in names:
        assert hasattr(lib, n), n


def test_abi_version_and_error_string(lib):
    assert lib.mlstm_b200_abi_version() == 4
    assert isinstance(lib.mlstm_b200_last_error(), bytes)


def test_struct_sizes_match_header(lib):
    """Compile a tiny C program against the header and compare sizeof with the ctypes mirror."""
    import subprocess
    import tempfile

    from xlstm_yolo_clean_b200 import _cabi

    code = '#include <stdio.h>\n#include "mlstm_b200.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n",' \
           "sizeof(mlstm_b200_tensor),sizeof(mlstm_b200_shape),sizeof(mlstm_b200_fw_args),sizeof(mlstm_b200_bw_args)," \
           "sizeof(mlstm_b200_cellout_args),sizeof(mlstm_b200_cellout_bw_args)," \
           "sizeof(mlstm_b200_rmsnorm_args),sizeof(mlstm_b200_rmsnorm_bw_args),sizeof(mlstm_b200_recurrent_args),sizeof(mlstm_b200_fw_epilogue));}"
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "s.c")
        open(c, "w").write(code)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", os.path.join(d, "s")])
        out = subprocess.check_output([os.path.join(d, "s")]).split()
    sizes = [int(x) for x in out]
    assert sizes == [ctypes.sizeof(_cabi.Tensor), ctypes.sizeof(_cabi.Shape), ctypes.sizeof(_cabi.FwArgs),
                     ctypes.sizeof(_cabi.BwArgs), ctypes.sizeof(_cabi.CellOutArgs), ctypes.sizeof(_cabi.CellOutBwArgs),
                     ctypes.sizeof(_cabi.RmsNormArgs), ctypes.sizeof(_cabi.RmsNormBwArgs), ctypes.sizeof(_cabi.RecurrentArgs), ctypes.sizeof(_cabi.FwEpilogue)]


def test_workspace_query_needs_no_gpu(lib):
    from xlstm_yolo_clean_b200 import _cabi

    s = _cabi.Shape()
    s.B, s.NH, s.S, s.DHQK, s.DHHV, s.chunk_size, s.dtype, s.impl = 2, 4, 256, 64, 64, 64, _cabi.F32, _cabi.IMPL_EXACT
    fw = lib.mlstm_b200_workspace_bytes(ctypes.byref(s), 0)
    bw = lib.mlstm_b200_workspace_bytes(ctypes.byref(s), 1)
    assert 0 < fw < bw


def test_cpu_tensors_are_refused():
    import xlstm_yolo_clean_b200 as pkg

    q = torch.randn(1, 1, 64, 16)
    g = torch.randn(1, 1, 64)
    with pytest.raises(RuntimeError, match="no CPU path"):
        pkg.mlstm_chunkwise__b200(q=q, k=q, v=q, i=g, f=g)


def test_missing_library_fails_loudly(tmp_path):
    from xlstm_yolo_clean_b200 import _cabi

    with pytest.raises(_cabi.LibraryMissing):
        _cabi.load_library(str(tmp_path / "nope.so"))


def test_compute_call_without_device_returns_error(lib):
    """On a box without a GPU the compute entry points must return an error, never compute."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from xlstm_yolo_clean_b200 import _cabi

    a = _cabi.FwArgs()
    a.shape.B, a.shape.NH, a.shape.S, a.shape.DHQK, a.shape.DHHV, a.shape.chunk_size = 1, 1, 64, 16, 16, 64
    dummy = ctypes.create_string_buffer(64)
    p = ctypes.addressof(dummy)
    for t in (a.q, a.k, a.v, a.h, a.i, a.f):
        t.ptr = p
        t.stride[3] = 1
    a.n_out = a.m_out = p
    st = lib.mlstm_b200_chunkwise_fw(ctypes.byref(a), None)
    assert st != 0
    assert lib.mlstm_b200_last_error() != b""


def test_registry_drop_in():
    """register() makes 'chunkwise--b200' resolvable through the reference's get_mlstm_kernel
    (only where the reference is staged under baseline/_ref, tools/stage_reference.sh)."""
    import sys

    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref, "mlstm_kernels")):
        pytest.skip("reference not staged under baseline/_ref (tools/stage_reference.sh)")
    sys.path.insert(0, ref)
    sys.dont_write_bytecode = True
    try:
        import xlstm_yolo_clean_b200 as pkg
        from mlstm_kernels.torch import get_mlstm_kernel
        from mlstm_kernels.torch.backend_module import mLSTMBackend, mLSTMBackendConfig

        full = pkg.register()
        assert get_mlstm_kernel(full) is pkg.mlstm_chunkwise__b200
        be = mLSTMBackend(mLSTMBackendConfig(chunkwise_kernel=full, mode="train_with_padding", return_last_states=False))
        q = torch.randn(1, 2, 100, 16)
        g = torch.randn(1, 2, 100)
        with pytest.raises(RuntimeError, match="no CPU path"):  # routed to our kernel, which refuses CPU
            be(q=q, k=q, v=q, i=g, f=g)
    finally:
        sys.path.remove(ref)


def test_rotated_conv_equals_flip_conv_flip():
    """The identity the flip-free bottom-right branch rests on (vision_lstm2.py:292-294, 309-310): flipping the
    row-major token sequence is a 180-degree rotation of the image, so conv(flip(x)) flipped back equals the
    depthwise conv with its 3x3 kernel rotated.  Pure host logic, CPU."""
    from xlstm_yolo_clean_b200 import vil

    torch.manual_seed(0)
    conv = torch.nn.Conv2d(24, 24, 3, padding=1, groups=24).double()
    conv.seqlens = [6, 6]
    x = torch.randn(2, 36, 48, dtype=torch.float64)[..., :24]  # a chunk view, like x_qk in mlstm_branch
    want = vil._seq_conv(conv, x.flip(dims=[1]), rotate=False).flip(dims=[1])
    got = vil._seq_conv(conv, x, rotate=True)
    assert torch.allclose(got, want, atol=1e-12)


def test_fused_cell_refuses_cpu():
    import xlstm_yolo_clean_b200 as pkg

    with pytest.raises(RuntimeError, match="no CPU path"):
        pkg.cell_out(torch.randn(1, 4, 8, 64))


def test_cellout_without_device_returns_error(lib):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from xlstm_yolo_clean_b200 import _cabi

    a = _cabi.CellOutArgs()
    a.B, a.NH, a.S, a.D = 1, 2, 8, 64
    st = lib.mlstm_b200_cellout_fw(ctypes.byref(a), None)
    assert st != 0 and lib.mlstm_b200_last_error() != b""


class _PCell(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.dim, self.num_heads, self.gate_soft_cap = 256, 4, 15.0
        self.use_autocast, self.autocast_dtype = True, torch.float16
        self.ifgate = torch.nn.Linear(768, 8)

class _PLayer(torch.nn.Module):
    def __init__(self, heads_ok=True):
        super().__init__()
        self.direction = "ROWWISE_FROM_BOT_RIGHT"
        self.proj_up = torch.nn.Linear(128, 512)
        self.conv = torch.nn.Conv2d(256, 256, 3, padding=1, groups=256)
        self.qk_proj, self.v_proj = torch.nn.Linear(256, 512), torch.nn.Linear(256, 256)
        self.mlstm_cell = _PCell()
        if not heads_ok:
            self.mlstm_cell.num_heads = 5  # 256 / 5: geometry the fused output kernel does not cover
        self.learnable_skip = torch.nn.Parameter(torch.ones(256))
        self.proj_down = torch.nn.Linear(256, 128)
        self.norm, self.ffn_norm = torch.nn.RMSNorm(256, eps=1e-6), torch.nn.RMSNorm(100, eps=1e-6)


def test_patch_layers_rebinds_without_a_gpu():
    """Host logic of the fused-layer rebinding (vil.patch_layers): ViLLayer-shaped modules get the new branch and
    norm forwards; the norm keeps working for CPU tensors (torch's own forward), the branch refuses them."""
    import xlstm_yolo_clean_b200 as pkg

    model = torch.nn.Sequential(_PLayer(), _PLayer(heads_ok=False), torch.nn.Linear(4, 4))
    assert pkg.patch_layers(model) == 1
    a, b = model[0], model[1]
    assert "mlstm_branch" in a.__dict__ and "mlstm_branch" not in b.__dict__
    assert "forward" in a.norm.__dict__ and "forward" not in a.ffn_norm.__dict__  # dim 100 is not covered
    x = torch.randn(2, 9, 256)
    assert torch.allclose(a.norm(x), torch.nn.functional.rms_norm(x, (256,), a.norm.weight, 1e-6))
    with pytest.raises(RuntimeError, match="no CPU path"):
        a.mlstm_branch(torch.randn(1, 16, 128))
    assert pkg.vil._is_reverse(a)


def test_patched_model_survives_deepcopy_and_torch_save(tmp_path):
    """The reference trainer checkpoints whole modules -- torch.save({'ema': deepcopy(ema).half(), ...}),
    ultralytics/engine/trainer.py:517-540 -- so a patched model must pickle, load back, and stay bound to ITSELF
    (not to the module it was copied from)."""
    import copy

    import xlstm_yolo_clean_b200 as pkg

    model = torch.nn.Sequential(_PLayer(), torch.nn.Linear(4, 4))
    assert pkg.patch_layers(model, siging=True) == 1
    path = tmp_path / "last.pt"
    torch.save({"model": copy.deepcopy(model).half(), "epoch": 3}, path)
    loaded = torch.load(path, weights_only=False)["model"]
    for m in (copy.deepcopy(model), loaded):
        layer = m[0]
        assert "mlstm_branch" in layer.__dict__ and "forward" in layer.norm.__dict__
        assert layer.mlstm_branch.args[0] is layer and layer.norm.forward.args[0] is layer.norm  # re-bound to the copy
        assert layer.mlstm_branch.keywords == {"siging": True, "kernel_dtype": "bfloat16", "one_launch": "auto"}
        x = torch.randn(2, 9, 256, dtype=layer.norm.weight.dtype)
        assert torch.allclose(layer.norm(x), torch.nn.functional.rms_norm(x, (256,), layer.norm.weight, 1e-6))
        with pytest.raises(RuntimeError, match="no CPU path"):
            layer.mlstm_branch(torch.randn(1, 16, 128, dtype=layer.norm.weight.dtype))


def test_graphed_patch_survives_deepcopy_and_torch_save(tmp_path):
    """patch_layers(graphs=True) binds a vil._GraphedBranch: it pickles without its CUDA graphs and stays bound to the
    copy it travels with."""
    import copy

    import xlstm_yolo_clean_b200 as pkg

    model = torch.nn.Sequential(_PLayer(), torch.nn.Linear(4, 4))
    assert pkg.patch_layers(model, graphs=True) == 1
    model[0].mlstm_branch._graphs["sentinel"] = object()  # stands for a built graph
    path = tmp_path / "last.pt"
    torch.save({"model": copy.deepcopy(model).half()}, path)
    loaded = torch.load(path, weights_only=False)["model"]
    for m in (copy.deepcopy(model), loaded):
        br = m[0].mlstm_branch
        assert br.layer is m[0] and br._graphs == {} and br.cfg[1:] == ("bfloat16", "auto")
        with pytest.raises(RuntimeError, match="no CPU path"):
            br(torch.randn(1, 16, 128, dtype=m[0].norm.weight.dtype))


def test_call_plan_table_is_bounded():
    """Callers with ever-changing shapes must not grow the per-thread plan table without bound."""
    import xlstm_yolo_clean_b200.backend as be

    d = be._plans()
    d.clear()
    for i in range(be._MAX_PLANS):
        d[("dummy", i)] = None
    assert len(be._plans()) == 0
