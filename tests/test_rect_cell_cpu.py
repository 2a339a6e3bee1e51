"""Layer-layout views of a cell whose q / k are narrower than v (rectangular heads), checked without a device:
``vil._heads`` splits qk (B, S, 2 NH DHQK) = [q | k] and v (B, S, NH DHHV) into (B, NH, S, D) views of the same
storage, and the one-launch policy for rectangular heads covers both supported pairs in both grad modes."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from xlstm_yolo_clean_b200 import vil  # noqa: E402


@pytest.mark.parametrize("DK,DV", [(32, 64), (64, 128), (64, 64)])
def test_heads_views_of_rectangular_layer_tensors(DK, DV):
    B, S, NH = 2, 12, 3
    qk = torch.randn(B, S, 2 * NH * DK)
    v = torch.randn(B, S, NH * DV)
    gates = torch.randn(B, S, 2 * NH)
    assert vil._head_dims(qk, v, NH) == (DK, DV)
    q, k, vv, i, f = vil._heads(qk, v, gates, NH)
    assert q.shape == k.shape == (B, NH, S, DK) and vv.shape == (B, NH, S, DV) and i.shape == f.shape == (B, NH, S)
    for t, base in ((q, qk), (k, qk), (vv, v), (i, gates), (f, gates)):
        assert t.untyped_storage().data_ptr() == base.untyped_storage().data_ptr()  # views, no copies
    assert torch.equal(q, qk[..., :NH * DK].reshape(B, S, NH, DK).transpose(1, 2))
    assert torch.equal(k, qk[..., NH * DK:].reshape(B, S, NH, DK).transpose(1, 2))
    assert torch.equal(vv, v.reshape(B, S, NH, DV).transpose(1, 2))
    assert k.stride() == q.stride() == (S * 2 * NH * DK, DK, 2 * NH * DK, 1)


def test_grad_dtype_takes_head_dims_from_qk_and_v():
    NH, S = 4, 8
    ins = (torch.float16,) * 3
    for DK, DV, ok in ((32, 64, True), (64, 128, True), (64, 64, True), (32, 128, False), (48, 96, False)):
        qk = torch.empty(1, S, 2 * NH * DK, dtype=torch.bfloat16)
        v = torch.empty(1, S, NH * DV, dtype=torch.bfloat16)
        assert vil._layer_grad_dtype(ins, torch.bfloat16, vil._head_dims(qk, v, NH), S) == (
            torch.float16 if ok else torch.bfloat16), (DK, DV)


def test_rect_one_launch_policy_covers_both_pairs_and_grad_modes():
    assert set(vil.RECT_ONE_LAUNCH) == {(dk, dv, g) for dk, dv in ((32, 64), (64, 128)) for g in (False, True)}
