"""Float64 reference of the sigmoid-input-gate mLSTM without its normaliser (``normalize=False``) for the tests, built
on the unchanged primitives of ``oracle/mlstm_oracle.py``.

Without the normaliser h is the numerator of the oracle's siging forward, q̄ᵀC_{k-1} + Σ_{s<=t} P_ts v_s (every max
state is 0), and the backward is the oracle's siging backward with dh used as it is: ``chunkwise_bw`` scales dh by
1 / (n_tok + eps), which is exactly 1 for n_tok = 1 and eps = 0, and eps enters nowhere else.  n_out / m_out and the
states are those of the normalised call."""
import torch

from oracle import mlstm_oracle as O


def chunkwise_fw(q, k, v, i, f, c0=None, n0=None, chunk_size=64, eps=1e-6):
    """Returns h, n_out, m_out, (C_last, n_last, m_last) like ``O.chunkwise_fw(..., siging=True)``, h unnormalised."""
    B, NH, S, DK = q.shape
    DV = v.shape[-1]
    L, NC = chunk_size, S // chunk_size
    _, n_tok, m_tok, last, (C, _, _) = O.chunkwise_fw(q, k, v, i, f, c0, n0, None, chunk_size, eps, siging=True)
    gates = O.chunk_gates(i, f, L, siging=True)
    scale = DK ** -0.5
    qc, kc, vc = q.reshape(B, NH, NC, L, DK), k.reshape(B, NH, NC, L, DK), v.reshape(B, NH, NC, L, DV)
    p = torch.einsum("bhctd,bhcsd->bhcts", qc, kc) * scale * torch.exp(O._log_decay_matrix(gates))
    qbar = qc * (torch.exp(gates.b) * scale)[..., None]
    h = torch.einsum("bhctd,bhcde->bhcte", qbar, C[:, :, :NC]) + torch.einsum("bhcts,bhcse->bhcte", p, vc)
    return h.reshape(B, NH, S, DV), n_tok, m_tok, last


def chunkwise_bw(q, k, v, i, f, dh, c0=None, n0=None, dc_last=None, chunk_size=64):
    """dq, dk, dv, di, df, dC_initial of the unnormalised forward (never reads n_out)."""
    B, NH, S, _ = q.shape
    ones = torch.ones(B, NH, S, dtype=q.dtype)
    zeros = torch.zeros(B, NH, S, dtype=q.dtype)
    return O.chunkwise_bw(q, k, v, i, f, dh, ones, zeros, c0, n0, None, dc_last, chunk_size, eps=0.0, siging=True)


def fwbw(q, k, v, i, f, dh, c0=None, n0=None, dc_last=None, chunk_size=64, eps=1e-6):
    h, _, _, last = chunkwise_fw(q, k, v, i, f, c0, n0, chunk_size, eps)
    return h, last, chunkwise_bw(q, k, v, i, f, dh, c0, n0, dc_last, chunk_size)
