#!/usr/bin/env python
"""Sigmoid-input-gate mLSTM with and without the normaliser (normalize=True / False): device time of one forward and
one backward call on the tensor-core route (bf16) and on the exact fp32 FFMA route, at the config-2 call
(B=32 NH=4 S=1600 D=64) and a base192 call (768 heads = B 64 x NH 12, S=1600, D=32).  One JSON line per (shape, route)
on stdout and, with --out, appended to that file.

Timing: the period of back-to-back launches of one call captured in one CUDA graph, read with CUDA events
(rect_bench.graph_period_ms: best of three replays).  The two modes are measured alternately, --rounds times each; the
line reports each mode's best and the spread (max - min) over its rounds, so a difference can be read against the
run-to-run noise.  Inputs are the SURVEY.md section 8(d) config-2 distribution; `working_set_mb` says whether they fit
the 126 MB L2 (no flush between launches).  The GPU name and power limit are read in the same run.

    python tools/siging_norm_bench.py --out /tmp/siging_norm_bench.jsonl"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from rect_bench import call_bytes, gpu_info, graph_period_ms  # noqa: E402

SHAPES = [("config2", 32, 4, 1600, 64), ("base192", 64, 12, 1600, 32)]
ROUTES = [("tensor", torch.bfloat16, 8), ("exact", torch.float32, 2)]  # (route, dtype, launches per graph)


def inputs(B, NH, S, D, dtype, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    t = {k: torch.randn(B, NH, S, D, generator=g, device=dev).to(dtype) for k in ("q", "k", "v", "dh")}
    t["i"] = torch.randn(B, NH, S, generator=g, device=dev).to(dtype)
    t["f"] = (3.0 + torch.randn(B, NH, S, generator=g, device=dev)).to(dtype)
    return t


def calls(pkg, t, normalize):
    kw = dict(chunk_size=64, siging=True, normalize=normalize)
    fw = lambda: pkg.mlstm_chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], **kw)  # noqa: E731
    h, n_out, m_out, _, cst = fw()
    n_fw = pkg.last_launch_count()
    bw = lambda: pkg.mlstm_chunkwise_bw(t["q"], t["k"], t["v"], t["i"], t["f"], n_out, m_out, t["dh"],  # noqa: E731
                                        c_states=cst, **kw)
    bw()
    return fw, bw, n_fw, pkg.last_launch_count()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    ap.add_argument("--rounds", type=int, default=3, help="alternating measurements of each mode")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("siging_norm_bench.py needs a CUDA device")
    import __graft_entry__ as G

    G.build()
    import xlstm_yolo_clean_b200 as pkg

    dev = torch.device("cuda:0")
    name, power_w = gpu_info(dev)
    lines = []
    for tag, B, NH, S, D in SHAPES:
        for route, dtype, reps in ROUTES:
            t = inputs(B, NH, S, D, dtype, dev, seed=S + D)
            pkg.set_default_impl(route)
            try:
                fns = {nz: calls(pkg, t, nz) for nz in (True, False)}
                times = {nz: {"fw": [], "bw": []} for nz in (True, False)}
                for _ in range(args.rounds):
                    for nz in (True, False):
                        times[nz]["fw"].append(graph_period_ms(fns[nz][0], reps, dev))
                        times[nz]["bw"].append(graph_period_ms(fns[nz][1], reps, dev))
            finally:
                pkg.set_default_impl("auto")
            fwb, bwb = call_bytes(B, NH, S, D, D, t["q"].element_size())
            row = {"tool": "siging_norm_bench", "gpu": name, "power_limit_w": power_w, "shape": tag,
                   "B": B, "NH": NH, "S": S, "DHQK": D, "DHHV": D, "chunk_size": 64, "route": route,
                   "dtype": str(dtype).replace("torch.", ""), "working_set_mb": round((fwb + bwb) / 2 / 1e6, 1)}
            for nz, key in ((True, "normalize"), (False, "no_normalize")):
                fw, bw = times[nz]["fw"], times[nz]["bw"]
                row[key] = {"fw_us": min(fw) * 1e3, "bw_us": min(bw) * 1e3,
                            "fw_spread_us": (max(fw) - min(fw)) * 1e3, "bw_spread_us": (max(bw) - min(bw)) * 1e3,
                            "launches_fw": fns[nz][2], "launches_bw": fns[nz][3]}
            row["no_normalize_over_normalize"] = {
                "fw": row["no_normalize"]["fw_us"] / row["normalize"]["fw_us"],
                "bw": row["no_normalize"]["bw_us"] / row["normalize"]["bw_us"]}
            row["timing"] = (f"CUDA events around a graph of {reps} back-to-back launches of one call, best of 3 replays, "
                             f"modes alternated {args.rounds} times; no L2 flush")
            print(json.dumps(row), flush=True)
            lines.append(row)
            del t, fns
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as fh:
            for row in lines:
                fh.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
