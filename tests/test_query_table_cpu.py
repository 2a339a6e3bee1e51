"""The complete answer table of the host-only shape queries, without a device: tensor_path_supported, states_bytes and
workspace_bytes (forward and backward) under IMPL_AUTO / IMPL_TENSOR / IMPL_EXACT, over every tensor-core head pair and
its neighbours, fp32 / bf16 / fp16, full and ragged S, S % 4 != 0, and two chunk sizes.  Every geometry the tensor-core
route knows shows up in these sizes, so a wrong route or workspace for any shape fails here.

Regenerate the golden (only when a change of the table is intended):  python tests/test_query_table_cpu.py
"""
import ctypes
import itertools
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import __graft_entry__ as G  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden", "host_queries.txt.gz")  # one row per shape: KEYS, then the four answers
KEYS = "DHQK DHHV dtype S chunk_size impl"
ANSWERS = "tensor_path_supported states_bytes workspace_bytes(fw) workspace_bytes(bw)"
DIMS = (32, 48, 64, 96, 128, 192, 256, 512)
SEQ = (100, 196, 198, 6400)
CHUNKS = (4, 64)
B, NH = 2, 3


def _table():
    G.build()
    import xlstm_yolo_clean_b200 as pkg

    C = pkg._cabi
    lib = pkg.load_library()
    keys, answers = [], []
    for dk, dv, dt, S, chunk, impl in itertools.product(DIMS, DIMS, (C.F32, C.BF16, C.F16), SEQ, CHUNKS,
                                                         (C.IMPL_AUTO, C.IMPL_TENSOR, C.IMPL_EXACT)):
        s = C.Shape()
        s.B, s.NH, s.S, s.DHQK, s.DHHV, s.chunk_size, s.dtype, s.impl = B, NH, S, dk, dv, chunk, dt, impl
        p = ctypes.byref(s)
        keys.append((dk, dv, dt, S, chunk, impl))
        answers.append((lib.mlstm_b200_tensor_path_supported(p), lib.mlstm_b200_states_bytes(p),
                        lib.mlstm_b200_workspace_bytes(p, 0), lib.mlstm_b200_workspace_bytes(p, 1)))
    return np.array([k + a for k, a in zip(keys, answers)], dtype=np.int64)


def test_host_query_table_matches_golden():
    got = _table()
    want = np.loadtxt(GOLDEN, dtype=np.int64)
    assert got.shape == want.shape
    np.testing.assert_array_equal(got[:, :6], want[:, :6])
    bad = np.nonzero((got != want).any(axis=1))[0]
    assert bad.size == 0, [(got[i, :6].tolist(), got[i, 6:].tolist(), want[i, 6:].tolist()) for i in bad[:10]]


if __name__ == "__main__":
    t = _table()
    np.savetxt(GOLDEN, t, fmt="%d", header=f"{KEYS} | {ANSWERS}")
    print(f"wrote {GOLDEN}: {len(t)} shapes")
