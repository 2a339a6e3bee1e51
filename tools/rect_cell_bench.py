#!/usr/bin/env python
"""The mLSTM cell forward for rectangular heads (DHQK, DHHV) = (32, 64) and (64, 128) as one launch against two: the
rectangular forward with the fused cell-output epilogue (tc_fw_rect<..., EPI>, two-CTA clusters: MultiHeadLayerNorm,
(B, NH, S, DHHV) -> (B, S, NH DHHV) relayout and learnable skip in the kernel) against the plain rectangular forward
followed by the stand-alone cell-output kernel (k_cellout_fw).  Both without gradients (y only) and in training (h and
the per-tile states also written, as the backward needs them), at B=32 NH=4 S=1600 and B=16 NH=6 S=6400; bf16 kernels,
fp16 y and skip input (ultralytics' AMP).  One JSON line per (pair, size, grad mode) on stdout and, with --out, appended
to that file.

Timing: the period of back-to-back launches of one cell forward captured in one CUDA graph, read with CUDA events, best
of three replays (tools/rect_bench.py); the two arms alternate (fused, two-launch, fused, two-launch) in the same run and
each reports its best round.  Their outputs on the same seeded inputs are compared (max|a-b| / max|b|; h must be
bit-identical).  `active_clusters` is cudaOccupancyMaxActiveClusters of the fused kernel; the GPU name and power limit
are read in the same run.

    python tools/rect_cell_bench.py --out /tmp/rect_cell_bench.jsonl"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from rect_bench import gpu_info, graph_period_ms  # noqa: E402

PAIRS = [(32, 64), (64, 128)]
SIZES = [(32, 4, 1600), (16, 6, 6400)]


def inputs(B, NH, S, DK, DV, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    H = NH * DV
    qk = (0.3 * torch.randn(B, S, 2 * NH * DK, generator=g, device=dev)).to(torch.bfloat16)
    v = (0.3 * torch.randn(B, S, H, generator=g, device=dev)).to(torch.bfloat16)
    gates = torch.cat([-6.0 + torch.randn(B, S, NH, generator=g, device=dev),
                       3.0 + 3.0 * torch.rand(B, S, NH, generator=g, device=dev)], -1).to(torch.bfloat16)
    x = torch.randn(B, S, H, generator=g, device=dev).to(torch.float16)
    w = 1.0 + 0.1 * torch.randn(H, generator=g, device=dev)
    b = 0.1 * torch.randn(H, generator=g, device=dev)
    sk = 1.0 + 0.1 * torch.randn(H, generator=g, device=dev)
    return qk, v, gates, x, w, b, sk


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", default=None, help="append the JSON lines to this file")
    ap.add_argument("--reps", type=int, default=8, help="cell forwards per CUDA graph")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("rect_cell_bench.py needs a CUDA device")
    import ctypes as C

    import __graft_entry__ as G

    G.build()
    import xlstm_yolo_clean_b200 as pkg
    from xlstm_yolo_clean_b200 import _cabi, backend

    dev = torch.device("cuda:0")
    name, power_w = gpu_info(dev)
    lib = _cabi.load_library()
    lines = []
    for DK, DV in PAIRS:
        for B, NH, S in SIZES:
            qk, v, gates, x, w, b, sk = inputs(B, NH, S, DK, DV, dev, seed=S + DK)
            q, k, vv, i, f = pkg.vil._heads(qk, v, gates, NH)
            H = NH * DV
            heads = lambda t: t.view(B, S, NH, DV).transpose(1, 2)  # noqa: E731
            shape = backend._shape(q, vv, 64, 1e-6, None)
            clusters = lib.mlstm_b200_debug_fw_epilogue_clusters(C.byref(shape))
            for train in (False, True):
                y = torch.empty(B, S, H, dtype=torch.float16, device=dev)

                def fused():
                    epi = backend.FwEpilogue(heads(y), heads(x), w, b, sk, 1e-6, train)
                    return backend._fw_launch(q, k, vv, i, f, None, None, None, None, False, 64, 1e-6, None, train,
                                              False, False, 0.0, epi)[0], y

                def two_launch():
                    h = backend._fw_launch(q, k, vv, i, f, None, None, None, None, False, 64, 1e-6, None, train, False,
                                           False, 0.0)[0]
                    return h, pkg.cell_out(h, w, b, sk, x, eps=1e-6, out_dtype=torch.float16)

                with torch.no_grad():
                    h_f, y_f = fused()
                    n_fused = pkg.last_launch_count()
                    y_f = y_f.clone()
                    h_t, y_t = two_launch()
                    torch.cuda.synchronize()
                    err = float((y_f.float() - y_t.float()).abs().max() / y_t.float().abs().max())
                    h_equal = None if h_f is None else bool(torch.equal(h_f, h_t))
                    t_f, t_t = [], []
                    for _ in range(2):  # alternate the arms
                        t_f.append(graph_period_ms(fused, args.reps, dev))
                        t_t.append(graph_period_ms(two_launch, args.reps, dev))
                row = {
                    "tool": "rect_cell_bench", "gpu": name, "power_limit_w": power_w, "kernel_dtype": "bf16",
                    "y_dtype": "fp16", "B": B, "NH": NH, "S": S, "DHQK": DK, "DHHV": DV,
                    "mode": "training (h and states written)" if train else "no-grad (y only)",
                    "fused_us": min(t_f) * 1e3, "two_launch_us": min(t_t) * 1e3,
                    "fused_over_two_launch": min(t_f) / min(t_t),
                    "rounds_us": {"fused": [t * 1e3 for t in t_f], "two_launch": [t * 1e3 for t in t_t]},
                    "launches_fused": n_fused, "active_clusters": clusters, "clusters_in_grid": B * NH,
                    "y_max_rel_diff": err, "h_bit_identical": h_equal,
                    "timing": f"CUDA events around a graph of {args.reps} back-to-back cell forwards, best of 3 replays, "
                              "/ launches; arms alternated twice, best round",
                }
                print(json.dumps(row), flush=True)
                lines.append(row)
            del qk, v, gates, x
            torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as fh:
            for row in lines:
                fh.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
