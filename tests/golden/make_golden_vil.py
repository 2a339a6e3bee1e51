"""Golden vectors of the UNMODIFIED reference ViLLayer.mlstm_branch (staged under baseline/_ref by tools/stage_reference.sh).

    PYTHONDONTWRITEBYTECODE=1 YOLO_CONFIG_DIR=/tmp/yolo_cfg python tests/golden/make_golden_vil.py

Builds the reference's own ``ViLLayer`` (ultralytics/nn/modules/vision_lstm/vision_lstm2.py:218-351) on the CPU in
float64 -- where ``MatrixLSTMCell`` selects ``chunkwise--native_autograd`` (:670-682, :708) -- for both scan
directions, perturbs the parameters the reference initialises to trivial values (ifgate weight = 0, outnorm weight
= 0), and records: every parameter of the branch, an input x, ``layer.mlstm_branch(x)`` (flips, SequenceConv2d,
qk/v projections, the cell with MultiHeadLayerNorm, learnable skip, proj_down) and the gradient of a fixed
cotangent w.r.t. x.  tests/test_cell_gpu.py::test_branch_matches_reference_vil_layer_golden loads the parameters
into an attribute-compatible stand-in and requires ``mlstm_branch_b200`` (no flips, anti-causal kernel, rotated conv,
fused cell output) to reproduce them on the GPU.
"""
import os
import sys
import types

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "..", "baseline", "_ref"))
sys.dont_write_bytecode = True
os.environ.setdefault("YOLO_CONFIG_DIR", "/tmp/yolo_cfg")
for name in ("matplotlib", "matplotlib.pyplot"):
    sys.modules.setdefault(name, types.ModuleType(name))
sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]

from ultralytics.nn.modules.vision_lstm.vision_lstm2 import SequenceTraversal, ViLLayer  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
DIM, QKV_BLOCK, SIDE, B = 64, 32, 10, 2  # inner 128, NH = 4, D = 32; S = 100: the padded stage of the models


def make(tag, direction, side, seed, w_mul, gate_std, norm_mean, suffix=""):
    torch.manual_seed(seed)
    layer = ViLLayer(dim=DIM, direction=direction, qkv_block_size=QKV_BLOCK, seqlens=[side, side], chunk_size=64).double()
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        cell = layer.mlstm_cell
        cell.ifgate.weight.copy_(gate_std * torch.randn(cell.ifgate.weight.shape, generator=g, dtype=torch.float64))
        cell.ifgate.bias[: cell.num_heads] = -2.0  # input gates that matter (the reference's -10 mutes the recurrence)
        cell.outnorm.weight.copy_(norm_mean + 0.2 * torch.randn(cell.outnorm.weight.shape, generator=g, dtype=torch.float64))
        if cell.outnorm.bias is not None:
            cell.outnorm.bias.copy_(0.1 * torch.randn(cell.outnorm.bias.shape, generator=g, dtype=torch.float64))
        layer.learnable_skip.copy_(1.0 + 0.2 * torch.randn(layer.learnable_skip.shape, generator=g, dtype=torch.float64))
        for lin in (layer.proj_up, layer.qk_proj, layer.v_proj, layer.proj_down):  # small_init_ leaves them tiny
            lin.weight.mul_(w_mul)
    x = torch.randn(B, side * side, DIM, generator=g, dtype=torch.float64).requires_grad_(True)
    dout = torch.randn(B, side * side, DIM, generator=g, dtype=torch.float64)
    layer.train()
    y = layer.mlstm_branch(x)
    (dx,) = torch.autograd.grad(y, x, dout)
    keep = ("proj_up", "conv", "qk_proj", "v_proj", "mlstm_cell.ifgate", "mlstm_cell.outnorm", "learnable_skip", "proj_down")
    out = {"p_" + k: v.detach().numpy() for k, v in layer.state_dict().items() if k.startswith(keep)}
    out.update(x=x.detach().numpy(), dout=dout.numpy(), y=y.detach().numpy(), dx=dx.numpy(),
               meta=np.array([DIM, layer.num_heads, side, B]))
    path = os.path.join(HERE, f"vil_layer_{suffix}{tag}.npz")
    np.savez_compressed(path, **out)
    print(suffix + tag, "->", path, {k: v.shape for k, v in out.items() if k.startswith("p_")}, "|y|max", float(y.abs().max()))


def main():
    for tag, direction in (("fwd", SequenceTraversal.ROWWISE_FROM_TOP_LEFT), ("rev", SequenceTraversal.ROWWISE_FROM_BOT_RIGHT)):
        # the round-1 vectors: S = 100, tiny projections -> h has a small per-head variance (16-bit rounding of h is
        # amplified by the LayerNorm behind it: only the fp32 kernels are held tightly on them)
        make(tag, direction, SIDE, 11, 4.0, 0.05, 0.0)
        # well-conditioned vectors: S = 144 (one full 128-token tile + a ragged one), q / k / v of order 1-10 and gate
        # pre-activations spread like a trained model's (i in [-4, 0], f in [1, 7]) -> rounding q/k/v/i/f/h to fp16
        # inside the reference itself moves y and dx by 7e-4 (measured), so the 16-bit tensor-core path is held on
        # output AND input gradient.  (Wider gates or larger projections make h = num / max(|q.n|, e^-m) spike to
        # 1e3-1e5 at single tokens, beyond what an fp16 h can carry -- in the reference's own fp16 rule as well.)
        make(tag, direction, 12, 21, 2.0, 0.02, 1.0, suffix="wc_")


if __name__ == "__main__":
    main()
