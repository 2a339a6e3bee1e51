"""Generate golden vectors from the UNMODIFIED reference.

    sh tools/stage_reference.sh <checkout of xlstm-yolo-clean>
    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py

Imports ``mlstm_kernels`` from the staged copy under baseline/_ref (read-only; the
repository does not carry the reference, which is why the outputs are committed as
``tests/golden/*.npz``).  Every case runs the reference in float64 on seeded inputs:

  * ``mlstm_chunkwise__native_custbw`` through autograd (the user-facing API whose
    backward is the spec, native/fwbw.py:228-263) -> h, last states, dq dk dv di df dc0
  * ``mlstm_chunkwise_fw`` directly (native/fw.py:224-318) -> n_out, m_out
  * ``wrap_chunkwise__pad_zeros`` (kernel_wrappers.py:204-265) for the ragged case
  * ``mlstm_recurrent_sequence__native_fw`` is not used; the oracle carries its own
    step recurrence and is checked against these vectors instead.
"""

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
sys.path.insert(0, os.path.join(HERE, "..", "..", "baseline", "_ref"))
sys.dont_write_bytecode = True

from mlstm_kernels.torch import get_mlstm_kernel  # noqa: E402
from mlstm_kernels.torch.chunkwise.native.fw import mlstm_chunkwise_fw  # noqa: E402
from mlstm_kernels.torch.kernel_wrappers import wrap_chunkwise__pad_zeros  # noqa: E402

from oracle.mlstm_oracle import make_inputs  # noqa: E402  (input generator only)

CASES = {
    # name: (B, NH, S, DK, DV, L, dist, with_states, seed)
    "plain_L64": (2, 2, 128, 16, 16, 64, "normal", False, 0),
    "states_L64": (1, 2, 192, 16, 16, 64, "normal", True, 1),
    "rect_L32": (1, 2, 96, 16, 32, 32, "normal", True, 2),
    "model_L64": (1, 3, 128, 32, 32, 64, "model", False, 3),
    "long_L64": (1, 1, 512, 16, 16, 64, "normal", False, 4),
}


def run_case(name, B, NH, S, DK, DV, L, dist, with_states, seed):
    inp = make_inputs(B, NH, S, DK, DV, seed=seed, dtype=torch.float64, dist=dist, with_states=with_states)
    leaf = {k: inp[k].clone().requires_grad_(True) for k in ("q", "k", "v", "i", "f")}
    c0 = inp.get("c0")
    if c0 is not None:
        c0 = c0.clone().requires_grad_(True)
    n0, m0 = inp.get("n0"), inp.get("m0")
    fn = get_mlstm_kernel("chunkwise--native_custbw")
    out = fn(q=leaf["q"], k=leaf["k"], v=leaf["v"], i=leaf["i"], f=leaf["f"], c_initial=c0, n_initial=n0,
             m_initial=m0, return_last_states=with_states, eps=1e-6, chunk_size=L,
             autocast_kernel_dtype=torch.float32)  # cast only applies under CUDA autocast
    if with_states:
        h, (c_last, n_last, m_last) = out
        (h * inp["dh"]).sum().add((c_last * inp["dc_last"]).sum()).backward()
    else:
        h = out
        (h * inp["dh"]).sum().backward()
    with torch.no_grad():
        _, n_out, m_out, _, _ = mlstm_chunkwise_fw(
            matQ=inp["q"], matK=inp["k"], matV=inp["v"], vecI=inp["i"], vecF=inp["f"], matC_initial=inp.get("c0"),
            vecN_initial=n0, scaM_initial=m0, chunk_size=L, eps=1e-6)
    blob = {f"in_{k}": v.numpy() for k, v in inp.items()}
    blob.update(h=h.detach().numpy(), n_out=n_out.numpy(), m_out=m_out.numpy(),
                dq=leaf["q"].grad.numpy(), dk=leaf["k"].grad.numpy(), dv=leaf["v"].grad.numpy(),
                di=leaf["i"].grad.numpy(), df=leaf["f"].grad.numpy(),
                meta=np.array([B, NH, S, DK, DV, L, int(with_states), seed]))
    if with_states:
        blob.update(c_last=c_last.detach().numpy(), n_last=n_last.detach().numpy(), m_last=m_last.detach().numpy(),
                    dc0=c0.grad.numpy())
    np.savez_compressed(os.path.join(HERE, f"{name}.npz"), **blob)
    print(name, "h", tuple(h.shape), "|h|max", float(h.abs().max()))


def run_padded():
    """S=100 is padded to 128 by the reference wrapper (kernel_wrappers.py:227-264)."""
    B, NH, S, DK, DV = 1, 2, 100, 16, 16
    inp = make_inputs(B, NH, S, DK, DV, seed=5, dtype=torch.float64)
    leaf = {k: inp[k].clone().requires_grad_(True) for k in ("q", "k", "v", "i", "f")}
    fn = get_mlstm_kernel("chunkwise--native_custbw")
    h = wrap_chunkwise__pad_zeros(fn, q=leaf["q"], k=leaf["k"], v=leaf["v"], i=leaf["i"], f=leaf["f"])
    (h * inp["dh"]).sum().backward()
    blob = {f"in_{k}": v.numpy() for k, v in inp.items()}
    blob.update(h=h.detach().numpy(), dq=leaf["q"].grad.numpy(), dk=leaf["k"].grad.numpy(),
                dv=leaf["v"].grad.numpy(), di=leaf["i"].grad.numpy(), df=leaf["f"].grad.numpy(),
                meta=np.array([B, NH, S, DK, DV, 64, 0, 5]))
    np.savez_compressed(os.path.join(HERE, "padded_S100.npz"), **blob)
    print("padded_S100", tuple(h.shape))


def run_siging():
    """Sigmoid-input-gate variant (what the reference's CUDA model path computes, vision_lstm2.py:685-697):
    quadratic native formulation ``parallel--native_siging_custbw`` (n treated as a constant in the backward,
    parallel/native_siging/bw.py), float64."""
    B, NH, S, DK, DV = 1, 2, 192, 16, 32
    inp = make_inputs(B, NH, S, DK, DV, seed=6, dtype=torch.float64)
    leaf = {k: inp[k].clone().requires_grad_(True) for k in ("q", "k", "v", "i", "f")}
    fn = get_mlstm_kernel("parallel--native_siging_custbw")
    h = fn(q=leaf["q"], k=leaf["k"], v=leaf["v"], i=leaf["i"], f=leaf["f"], eps=1e-6)
    (h * inp["dh"]).sum().backward()
    blob = {f"in_{k}": v.numpy() for k, v in inp.items()}
    blob.update(h=h.detach().numpy(), dq=leaf["q"].grad.numpy(), dk=leaf["k"].grad.numpy(),
                dv=leaf["v"].grad.numpy(), di=leaf["i"].grad.numpy(), df=leaf["f"].grad.numpy(),
                meta=np.array([B, NH, S, DK, DV, 64, 0, 6]))
    np.savez_compressed(os.path.join(HERE, "siging_S192.npz"), **blob)
    print("siging_S192", tuple(h.shape))


if __name__ == "__main__":
    torch.set_default_dtype(torch.float64)  # reference allocates its state buffers in the input dtype anyway
    for name, cfg in CASES.items():
        run_case(name, *cfg)
    run_padded()
    run_siging()
