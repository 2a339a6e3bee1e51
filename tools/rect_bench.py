#!/usr/bin/env python
"""Rectangular heads (DHQK, DHHV) = (32, 64) and (64, 128), bf16: device time of one forward and one backward call on
the tensor-core route (tc_fw_rect, two tc_bw<DHQK> block problems) and on the exact fp32 FFMA route that such calls
took before, at the two BASELINE call sizes B=32 NH=4 S=1600 and B=16 NH=6 S=6400, next to the square forward at
DHQK = DHHV = the same DHHV.  One JSON line per (pair, size) on stdout and, with --out, appended to that file.

Timing: the period of back-to-back launches of one call captured in one CUDA graph, read with CUDA events (the method
of bench.py's roofline block), best of three replays.  The same inputs are reused by every launch; `working_set_mb`
says whether they fit the 126 MB L2.  Bandwidth: algorithmic bytes (every input read once, every output written once,
the saved c_states excluded) over the device time, and its fraction of the measured 6535.7 GB/s copy peak of the B200
(SURVEY.md).  The GPU name and power limit are read in the same run.  `max_rel_err_vs_exact` compares the two routes'
outputs (max|a-b| / max|b| per tensor).

    python tools/rect_bench.py --out /tmp/rect_bench.jsonl"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_PEAK_GBS = 6535.7
PAIRS = [(32, 64), (64, 128)]
SIZES = [(32, 4, 1600), (16, 6, 6400)]


def call_bytes(B, NH, S, DK, DV, itemsize=2):
    tok = B * NH * S
    fw = tok * ((2 * DK + 2 * DV) * itemsize + 2 * itemsize + 8)  # read q, k, v, i, f; write h, n_out, m_out
    bw = tok * ((4 * DK + 3 * DV) * itemsize + 4 * itemsize + 8)  # read q, k, v, dh, i, f, n, m; write dq, dk, dv, di, df
    return fw, bw


def graph_period_ms(fn, reps, dev):
    keep = []
    side = torch.cuda.Stream(dev)
    with torch.cuda.stream(side):
        fn()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            for _ in range(reps):
                keep.append(fn())
    torch.cuda.synchronize()
    g.replay()
    ts = []
    for _ in range(3):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        g.replay()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) / reps)
    del g, keep
    return min(ts)


def gpu_info(dev):
    name = torch.cuda.get_device_name(dev)
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(dev.index or 0)
        return name, pynvml.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0
    except Exception:
        pass
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", str(dev.index or 0)],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return name, float(out.splitlines()[0])
    except Exception:
        return name, None


def inputs(B, NH, S, DK, DV, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    t = {k: (0.3 * torch.randn(B, NH, S, DK, generator=g, device=dev)).to(torch.bfloat16) for k in ("q", "k")}
    t.update({k: (0.3 * torch.randn(B, NH, S, DV, generator=g, device=dev)).to(torch.bfloat16) for k in ("v", "dh")})
    t["i"] = (-6.0 + torch.randn(B, NH, S, generator=g, device=dev)).to(torch.bfloat16)
    t["f"] = (3.0 + 3.0 * torch.rand(B, NH, S, generator=g, device=dev)).to(torch.bfloat16)
    return t


def route(pkg, t, impl, dev, reps):
    """fw / bw device time of one call and its outputs, on route `impl`."""
    pkg.set_default_impl(impl)
    try:
        fw = lambda: pkg.mlstm_chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=64)  # noqa: E731
        h, n_out, m_out, _, cst = fw()
        n_fw = pkg.last_launch_count()
        bw = lambda: pkg.mlstm_chunkwise_bw(t["q"], t["k"], t["v"], t["i"], t["f"], n_out, m_out, t["dh"],  # noqa: E731
                                            chunk_size=64, c_states=cst)
        grads = bw()
        n_bw = pkg.last_launch_count()
        fw_ms = graph_period_ms(fw, reps, dev)
        bw_ms = graph_period_ms(bw, reps, dev)
    finally:
        pkg.set_default_impl("auto")
    outs = dict(h=h, dq=grads[0], dk=grads[1], dv=grads[2], di=grads[3], df=grads[4])
    return fw_ms, bw_ms, n_fw, n_bw, outs


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    ap.add_argument("--reps", type=int, default=8, help="launches per CUDA graph on the tensor route")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("rect_bench.py needs a CUDA device")
    import __graft_entry__ as G

    G.build()
    import xlstm_yolo_clean_b200 as pkg

    dev = torch.device("cuda:0")
    name, power_w = gpu_info(dev)
    lines = []
    for DK, DV in PAIRS:
        for B, NH, S in SIZES:
            assert pkg.tensor_path_supported(B, NH, S, DK, DV, torch.bfloat16)
            t = inputs(B, NH, S, DK, DV, dev, seed=S + DK)
            tc = route(pkg, t, "tensor", dev, args.reps)
            ex = route(pkg, t, "exact", dev, 2)
            sq = inputs(B, NH, S, DV, DV, dev, seed=S + DV)
            sq_fw_ms = graph_period_ms(lambda: pkg.mlstm_chunkwise_fw(sq["q"], sq["k"], sq["v"], sq["i"], sq["f"], chunk_size=64),
                                       args.reps, dev)
            del sq
            fwb, bwb = call_bytes(B, NH, S, DK, DV)
            err = {k: float((tc[4][k].float() - ex[4][k].float()).abs().max() / ex[4][k].float().abs().max()) for k in tc[4]}
            row = {
                "tool": "rect_bench", "gpu": name, "power_limit_w": power_w, "dtype": "bf16",
                "B": B, "NH": NH, "S": S, "DHQK": DK, "DHHV": DV, "chunk_size": 64,
                "working_set_mb": round((fwb + bwb) / 2 / 1e6, 1),
                "tensor": {"fw_us": tc[0] * 1e3, "bw_us": tc[1] * 1e3, "launches_fw": tc[2], "launches_bw": tc[3],
                           "fw_gbs": fwb / tc[0] / 1e6, "bw_gbs": bwb / tc[1] / 1e6,
                           "fw_frac_of_copy_peak": fwb / tc[0] / 1e6 / HBM_PEAK_GBS,
                           "bw_frac_of_copy_peak": bwb / tc[1] / 1e6 / HBM_PEAK_GBS},
                "exact": {"fw_us": ex[0] * 1e3, "bw_us": ex[1] * 1e3, "launches_fw": ex[2], "launches_bw": ex[3],
                          "fw_gbs": fwb / ex[0] / 1e6, "bw_gbs": bwb / ex[1] / 1e6,
                          "fw_frac_of_copy_peak": fwb / ex[0] / 1e6 / HBM_PEAK_GBS,
                          "bw_frac_of_copy_peak": bwb / ex[1] / 1e6 / HBM_PEAK_GBS},
                "speedup_fw": ex[0] / tc[0], "speedup_bw": ex[1] / tc[1],
                "square_fw_us_same_dhhv": sq_fw_ms * 1e3,
                "algorithmic_bytes": {"fw": fwb, "bw": bwb}, "copy_peak_gbs": HBM_PEAK_GBS,
                "max_rel_err_vs_exact": err,
                "timing": f"CUDA events around a graph of back-to-back launches of one call ({args.reps} tensor, 2 exact), "
                          "best of 3 replays, / launches",
            }
            print(json.dumps(row), flush=True)
            lines.append(row)
            del t, tc, ex
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as fh:
            for row in lines:
                fh.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
