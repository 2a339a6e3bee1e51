#!/usr/bin/env python
"""xLSTM-Large's head geometry (DHQK, DHHV) = (256, 512) in fp32 -- the model run without autocast -- on the exact (fp32
FFMA) route: device time of one forward (k_states + k_fw_h) and one backward (k_states + k_bw_dc + k_bw_dqkv + k_bw_df)
at B NH S = 1 8 8192 and 4 8 4096, next to the fp32 oracle port (the torch ops of the reference's native_custbw
formulation, oracle/mlstm_oracle.py, on the same GPU: what a user of native_custbw gets) and, for context, the bf16
tensor-core route at the same shape.  One JSON line per size on stdout and, with --out, appended to that file.

Timing: the period of back-to-back launches of one call captured in one CUDA graph, read with CUDA events, best of three
replays (both routes of this project); best of three eager calls between device syncs (oracle port).  Algorithmic
FLOPs: oracle.algorithmic_flops (SURVEY.md section 8(d), chunk 64).  No share of peak is given: the measuring guide
quotes no fp32 non-tensor peak.  `derived_fp32_ffma_ceiling_tflops` is SMs x 128 FP32 lanes x 2 FLOP x the maximum SM
clock, all read in the same run -- a derived figure, not a data-sheet one.  The GPU name and power limit are read in
the same run too.

    python tools/exact_wide_bench.py --out profiles/r10_exact_wide_bench.jsonl"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from rect_bench import gpu_info, graph_period_ms  # noqa: E402

DK, DV, L = 256, 512, 64
SIZES = [(1, 8, 8192), (4, 8, 4096)]


def inputs(B, NH, S, dev, seed, dtype):
    g = torch.Generator(device=dev).manual_seed(seed)
    t = {k: torch.randn(B, NH, S, DK, generator=g, device=dev).to(dtype) for k in ("q", "k")}
    t.update({k: torch.randn(B, NH, S, DV, generator=g, device=dev).to(dtype) for k in ("v", "dh")})
    t["i"] = torch.randn(B, NH, S, generator=g, device=dev).to(dtype)
    t["f"] = (3.0 + torch.randn(B, NH, S, generator=g, device=dev)).to(dtype)
    return t


def max_sm_clock_mhz(dev):
    out = subprocess.run(["nvidia-smi", "--query-gpu=clocks.max.sm", "--format=csv,noheader,nounits", "-i",
                          str(dev.index or 0)], capture_output=True, text=True, timeout=30).stdout.strip()
    return float(out)


def route_us(pkg, t, impl, dev, reps):
    """fw / bw device time (us) of one call on route `impl`, launch counts and workspace bytes."""
    pkg.set_default_impl(impl)
    try:
        fw = lambda: pkg.mlstm_chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=L)  # noqa: E731
        h, n_out, m_out, _, cst = fw()
        n_fw = pkg.last_launch_count()
        bw = lambda: pkg.mlstm_chunkwise_bw(t["q"], t["k"], t["v"], t["i"], t["f"], n_out, m_out, t["dh"],  # noqa: E731
                                            chunk_size=L, c_states=cst)
        bw()
        n_bw = pkg.last_launch_count()
        fw_ms = graph_period_ms(fw, reps, dev)
        bw_ms = graph_period_ms(bw, reps, dev)
    finally:
        pkg.set_default_impl("auto")
    return fw_ms * 1e3, bw_ms * 1e3, n_fw, n_bw


def workspace_bytes(pkg, B, NH, S, dtype):
    C = pkg._cabi
    s = C.Shape()
    s.B, s.NH, s.S, s.DHQK, s.DHHV, s.chunk_size, s.dtype, s.impl = B, NH, S, DK, DV, L, dtype, C.IMPL_EXACT
    lib = pkg.load_library()
    return lib.mlstm_b200_workspace_bytes(ctypes.byref(s), 0), lib.mlstm_b200_workspace_bytes(ctypes.byref(s), 1)


def oracle_port_us(t, reps=3):
    from oracle import mlstm_oracle as O

    def fw():
        return O.chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=L)

    h, n_tok, m_tok, _, _ = fw()

    def bw():
        O.chunkwise_bw(t["q"], t["k"], t["v"], t["i"], t["f"], t["dh"], n_tok, m_tok, chunk_size=L)

    out = []
    for fn in (fw, bw):
        fn()
        best = float("inf")
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            best = min(best, time.perf_counter() - t0)
        out.append(best * 1e6)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    ap.add_argument("--reps", type=int, default=2, help="launches per CUDA graph")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("exact_wide_bench.py needs a CUDA device")
    import __graft_entry__ as G

    G.build()
    import xlstm_yolo_clean_b200 as pkg
    from oracle import mlstm_oracle as O

    dev = torch.device("cuda:0")
    name, power_w = gpu_info(dev)
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    clk = max_sm_clock_mhz(dev)
    ceiling = sms * 128 * 2 * clk * 1e6 / 1e12
    lines = []
    for B, NH, S in SIZES:
        ffw, fbw = O.algorithmic_flops(B, NH, S, DK, DV, L)
        t = inputs(B, NH, S, dev, S, torch.float32)
        fw_us, bw_us, n_fw, n_bw = route_us(pkg, t, "auto", dev, args.reps)
        assert (n_fw, n_bw) == (2, 4), "fp32 (256, 512) must run on the exact route"
        port_fw_us, port_bw_us = oracle_port_us(t)
        ws_fw, ws_bw = workspace_bytes(pkg, B, NH, S, pkg._cabi.F32)
        del t
        torch.cuda.empty_cache()
        t16 = inputs(B, NH, S, dev, S, torch.bfloat16)
        tc_fw_us, tc_bw_us, _, _ = route_us(pkg, t16, "tensor", dev, args.reps)
        del t16
        torch.cuda.empty_cache()
        rate = lambda fl, us: fl / (us * 1e-6) / 1e12  # noqa: E731
        row = {
            "tool": "exact_wide_bench", "gpu": name, "power_limit_w": power_w, "sms": sms, "max_sm_clock_mhz": clk,
            "B": B, "NH": NH, "S": S, "DHQK": DK, "DHHV": DV, "chunk_size": L,
            "exact_fp32": {"fw_us": fw_us, "bw_us": bw_us, "launches_fw": n_fw, "launches_bw": n_bw,
                           "fw_tflops": rate(ffw, fw_us), "bw_tflops": rate(fbw, bw_us),
                           "fwbw_tflops": rate(ffw + fbw, fw_us + bw_us),
                           "workspace_bytes_fw": ws_fw, "workspace_bytes_bw": ws_bw},
            "oracle_port_fp32": {"fw_us": port_fw_us, "bw_us": port_bw_us,
                                 "fwbw_tflops": rate(ffw + fbw, port_fw_us + port_bw_us),
                                 "matmul_allow_tf32": torch.backends.cuda.matmul.allow_tf32},
            "speedup_fwbw_vs_port": (port_fw_us + port_bw_us) / (fw_us + bw_us),
            "tensor_bf16_context": {"fw_us": tc_fw_us, "bw_us": tc_bw_us,
                                    "fwbw_tflops": rate(ffw + fbw, tc_fw_us + tc_bw_us)},
            "algorithmic_flops": {"fw": ffw, "bw": fbw},
            "derived_fp32_ffma_ceiling_tflops": ceiling,
            "timing": f"exact / tensor: CUDA events around a graph of {args.reps} back-to-back launches of one call, best "
                      "of 3 replays, / launches; port: best of 3 eager calls, host clock around device syncs",
        }
        print(json.dumps(row), flush=True)
        lines.append(row)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as fh:
            for row in lines:
                fh.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
