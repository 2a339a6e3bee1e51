#!/usr/bin/env python
"""xLSTM-Large's head geometry (DHQK, DHHV) = (256, 512), bf16: device time of one forward (tc_fw_wide, one launch) and
one backward (4 x 8 tc_bw<64> block problems, 32 launches with the forward's saved states) on the tensor-core route, at
B NH S = 1 8 8192 and 4 8 4096, next to the oracle port (the torch ops of the reference's native_custbw formulation,
oracle/mlstm_oracle.py, in bf16 on the same GPU).  One JSON line per size on stdout and, with --out, appended to that file.

Timing: the period of back-to-back launches of one call captured in one CUDA graph, read with CUDA events, best of three
replays (tensor route); best of three eager calls between CUDA events (oracle port).  Algorithmic FLOPs: SURVEY.md section
8(d) for DHQK != DHHV (oracle.algorithmic_flops, chunk 64); algorithmic bytes: every input read once, every output written
once, the saved c_states excluded.  `roof` says which roof binds at the call's arithmetic intensity (ridge = bf16 burst
peak / HBM copy peak of the B200) and the fraction of it reached.  The block-form backward reads q / k once per v block
(8 times) and v / dh once per qk block (4 times); `bw_block_bytes` counts that traffic (and the partial-sum read-backs of
the reduce-add stores and the c_states reads) against the algorithmic bytes.  The GPU name and power limit are read in
the same run.

    python tools/wide_bench.py --out profiles/r08_wide_bench.jsonl"""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from rect_bench import HBM_PEAK_GBS, call_bytes, gpu_info, graph_period_ms, inputs  # noqa: E402

BF16_PEAK_TFLOPS = 1652.1  # SURVEY.md: B200 bf16 dense burst
DK, DV = 256, 512
SIZES = [(1, 8, 8192), (4, 8, 4096)]


def block_bw_bytes(B, NH, S, bd=64, itemsize=2):
    """Bytes the 4 x 8 block problems move: each reads its bd-wide blocks of q, k, v, dh, the gates and n / m, and its
    block of c_states, writes its dq / dk / dv blocks (the later partials also read the earlier ones back: reduce-add)
    and di / df (read-modify-write after the first problem)."""
    tok, nq, nv = B * NH * S, DK // bd, DV // bd
    NT = (S + 127) // 128
    n = nq * nv
    reads = n * tok * (4 * bd * itemsize + 2 * itemsize + 8) + B * NH * NT * DK * DV * itemsize
    writes = n * tok * (3 * bd * itemsize + 2 * itemsize)
    readback = tok * bd * itemsize * (2 * nq * (nv - 1) + nv * (nq - 1)) + (n - 1) * tok * 2 * itemsize
    return reads + writes + readback


def roof(flops, nbytes, t_s):
    ai = flops / nbytes
    ridge = BF16_PEAK_TFLOPS * 1e12 / (HBM_PEAK_GBS * 1e9)
    t_roof = max(flops / (BF16_PEAK_TFLOPS * 1e12), nbytes / (HBM_PEAK_GBS * 1e9))
    return {"ai_flop_per_byte": ai, "ridge_flop_per_byte": ridge, "binds": "hbm" if ai < ridge else "tensor",
            "tflops": flops / t_s / 1e12, "gbs": nbytes / t_s / 1e9, "frac_of_roof": t_roof / t_s}


def oracle_port_ms(t, reps=3):
    from oracle import mlstm_oracle as O

    def step():
        h, n_tok, m_tok, _, _ = O.chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=64)
        O.chunkwise_bw(t["q"], t["k"], t["v"], t["i"], t["f"], t["dh"], n_tok, m_tok, chunk_size=64)

    def fw():
        O.chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=64)

    out = []
    for fn in (fw, step):
        fn()
        best = float("inf")
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            best = min(best, time.perf_counter() - t0)
        out.append(best * 1e3)
    return out[0], out[1] - out[0]  # fw, bw (fw + bw minus fw)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    ap.add_argument("--reps", type=int, default=4, help="launches per CUDA graph")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("wide_bench.py needs a CUDA device")
    import __graft_entry__ as G

    G.build()
    import xlstm_yolo_clean_b200 as pkg
    from oracle import mlstm_oracle as O

    dev = torch.device("cuda:0")
    name, power_w = gpu_info(dev)
    lines = []
    for B, NH, S in SIZES:
        assert pkg.tensor_path_supported(B, NH, S, DK, DV, torch.bfloat16)
        t = inputs(B, NH, S, DK, DV, dev, seed=S)
        fw = lambda: pkg.mlstm_chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=64)  # noqa: E731
        h, n_out, m_out, _, cst = fw()
        n_fw = pkg.last_launch_count()
        bw = lambda: pkg.mlstm_chunkwise_bw(t["q"], t["k"], t["v"], t["i"], t["f"], n_out, m_out, t["dh"],  # noqa: E731
                                            chunk_size=64, c_states=cst)
        bw()
        n_bw = pkg.last_launch_count()
        fw_ms = graph_period_ms(fw, args.reps, dev)
        bw_ms = graph_period_ms(bw, args.reps, dev)
        port_fw_ms, port_bw_ms = oracle_port_ms(t)
        ffw, fbw = O.algorithmic_flops(B, NH, S, DK, DV, 64)
        bfw, bbw = call_bytes(B, NH, S, DK, DV)
        blk = block_bw_bytes(B, NH, S)
        row = {
            "tool": "wide_bench", "gpu": name, "power_limit_w": power_w, "dtype": "bf16",
            "B": B, "NH": NH, "S": S, "DHQK": DK, "DHHV": DV, "chunk_size": 64,
            "tensor": {"fw_us": fw_ms * 1e3, "bw_us": bw_ms * 1e3, "launches_fw": n_fw, "launches_bw": n_bw,
                       "fw": roof(ffw, bfw, fw_ms * 1e-3), "bw": roof(fbw, bbw, bw_ms * 1e-3),
                       "fwbw": roof(ffw + fbw, bfw + bbw, (fw_ms + bw_ms) * 1e-3)},
            "oracle_port_bf16": {"fw_us": port_fw_ms * 1e3, "bw_us": port_bw_ms * 1e3,
                                 "fwbw_tflops": (ffw + fbw) / ((port_fw_ms + port_bw_ms) * 1e-3) / 1e12},
            "speedup_fwbw_vs_port": (port_fw_ms + port_bw_ms) / (fw_ms + bw_ms),
            "bw_share_of_fwbw": bw_ms / (fw_ms + bw_ms),
            "algorithmic_flops": {"fw": ffw, "bw": fbw}, "algorithmic_bytes": {"fw": bfw, "bw": bbw},
            "bw_block_bytes": blk, "bw_block_bytes_over_algorithmic": blk / bbw,
            "bw_block_bytes_gbs": blk / (bw_ms * 1e-3) / 1e9,
            "peaks": {"bf16_tflops": BF16_PEAK_TFLOPS, "hbm_gbs": HBM_PEAK_GBS},
            "timing": f"tensor: CUDA events around a graph of {args.reps} back-to-back launches of one call, best of 3 "
                      "replays, / launches; port: best of 3 eager calls, host clock around device syncs",
        }
        print(json.dumps(row), flush=True)
        lines.append(row)
        del t, h, n_out, m_out, cst
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as fh:
            for row in lines:
                fh.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
