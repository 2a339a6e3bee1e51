"""The host decisions the eager autograd Functions and the torch.compile ops share, checked without a device: the chunk
size / zero padding of a layer-layout call, the dtype the backward writes gradients in, and how the skip input of the
cell-output kernels is prepared (which inputs are copied)."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import __graft_entry__ as G  # noqa: E402

F16, BF16, F32 = torch.float16, torch.bfloat16, torch.float32
TENSOR_DIMS = [(32, 32), (64, 64), (128, 128), (32, 64), (64, 128)]
# S -> (chunk_size, pad) for chunk_size 64: 16-bit kernels on the tensor-core route run unpadded with gcd(S, 64)
ROUTE_PLAN = {100: (4, 0), 144: (16, 0), 400: (16, 0), 1600: (64, 0), 6400: (64, 0)}
PADDED_PLAN = {100: (64, 28), 144: (64, 48), 400: (64, 48), 1600: (64, 0), 6400: (64, 0)}


@pytest.fixture(scope="module")
def vil():
    G.build()
    from xlstm_yolo_clean_b200 import vil as v

    return v


@pytest.fixture
def exact_impl():
    from xlstm_yolo_clean_b200 import backend

    backend.set_default_impl("exact")
    yield
    backend.set_default_impl("auto")


@pytest.mark.parametrize("S", sorted(ROUTE_PLAN))
@pytest.mark.parametrize("DK,DV", TENSOR_DIMS + [(48, 96)])
@pytest.mark.parametrize("kdt", [BF16, F32])
def test_layer_chunking_and_grad_dtype(vil, S, DK, DV, kdt):
    NH = 4
    route = kdt is BF16 and (DK, DV) in TENSOR_DIMS
    chunk, pad = vil._layer_chunking(S, NH, (DK, DV), 64, kdt)
    assert (chunk, pad) == (ROUTE_PLAN if route else PADDED_PLAN)[S]
    # fp16 layer tensors: the bf16 tensor-core kernels write fp16 gradients themselves; elsewhere the kernel dtype
    assert vil._layer_grad_dtype((F16,) * 3, kdt, (DK, DV), S + pad) is (F16 if route else kdt)
    assert vil._layer_grad_dtype((BF16,) * 3, kdt, (DK, DV), S + pad) is (BF16 if kdt is BF16 else F32)
    assert vil._layer_grad_dtype((F16, F16, F32), kdt, (DK, DV), S + pad) is kdt  # no single caller dtype


@pytest.mark.parametrize("DK,DV", TENSOR_DIMS)
def test_grad_dtype_with_the_exact_kernels(vil, exact_impl, DK, DV):
    assert vil._layer_grad_dtype((F16,) * 3, BF16, (DK, DV), 1600) is BF16


def test_grad_dtype_rule_of_the_backward(vil):
    rule = vil._backend._grad_dtype
    assert rule(BF16, F16, True) is F16 and rule(F16, BF16, True) is BF16
    assert rule(BF16, F16, False) is BF16  # not the tensor-core route
    assert rule(BF16, None, True) is BF16 and rule(BF16, BF16, True) is BF16
    assert rule(BF16, F32, True) is BF16 and rule(F32, F16, False) is F32


def test_skip_input_preparation(vil):
    base = torch.randn(3 * 77 * 256 + 1, dtype=F16)
    aligned = base[:-1].view(3, 77, 256)
    assert vil._rows(aligned, F16) is aligned
    assert vil._rows(None, F16) is None
    for x in (base[1:].view(3, 77, 256),  # 2 bytes past an aligned base
              aligned.transpose(0, 1).contiguous().transpose(0, 1),  # permuted
              aligned.float()):  # wrong dtype
        y = vil._rows(x, F16)
        assert y.dtype is F16 and y.is_contiguous() and y.data_ptr() % 16 == 0 and y.untyped_storage().data_ptr() != \
            x.untyped_storage().data_ptr()
        assert torch.equal(y, x.to(F16))
