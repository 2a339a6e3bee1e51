"""The fused layer path at widths other than the three shipped YOLO-ViL ones (needs a B200).

One JSON line per measurement, each with the card name and power limit read in the same run:
  * copy_peak: a device-to-device copy of 4 GiB (read + write bytes over time): the HBM copy peak the kernel lines are
    measured against;
  * cellout_fw / cellout_bw at B = 32, S = 6400 for row widths H = NH * D with a tail warp (H mod 128 != 0) and for the
    128-multiple widths the shipped models use (the tail-free kernels): bf16 h, fp16 x / y / dy / dx, weight + bias +
    skip.  Algorithmic bytes: fw reads h, x and writes y (6 B per element); bw reads dy, h, x and writes dh, dx (10 B).
    Kernel time: the C-ABI call alone captured in a CUDA graph and replayed, the L2 flushed before every replay.  Next
    to it the torch composite it replaces (F.group_norm + relayout + skip add, autograd backward), eager, CUDA events;
  * rmsnorm_fw / rmsnorm_bw at 32 x 6400 rows of C channels, fp16 x / y / dy / dx and an fp32 weight (the fp16 autocast
    case): 4 B / 6 B per element; next to torch.rms_norm under fp16 autocast (its composite) and its autograd backward;
  * layer_step: one fp16-autocast training step (forward + backward) of a ViLLayer stand-in of width 320 (inner 640,
    5 heads of 128, both RMSNorms, FFN), B = 32, S = 6400, patched (patch_layers) vs unpatched (the reference's
    composition: flips, torch RMSNorm, group_norm, copies around the same mLSTM kernel).

    python tools/width_bench.py [--out profiles/r07_width_bench.jsonl] [--reps 20]
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import xlstm_yolo_clean_b200 as pkg  # noqa: E402
from xlstm_yolo_clean_b200 import vil  # noqa: E402

DEV = torch.device("cuda:0")
B, S = 32, 6400
TAIL_H = [(3, 32), (5, 32), (3, 64), (5, 64), (7, 64), (63, 32)]
WHOLE_H = [(6, 64), (8, 64), (12, 64), (5, 128), (16, 128)]
RMS_NEW = [64, 96, 128, 160, 320, 448, 640, 768, 1024, 2048]
RMS_SHIPPED = [192, 256, 384, 512]


def _card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else torch.cuda.get_device_name()


FLUSH = None


def _flush():
    FLUSH.zero_()  # 256 MB > the 126 MB L2: every timed pass reads its inputs from HBM


def graph_ms(fn, reps):
    """Median device time of fn's kernels alone: captured once in a CUDA graph, replayed after an L2 flush."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            keep = fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        _flush()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    del keep, g
    return sorted(ts)[len(ts) // 2]


def eager_ms(fn, reps):
    for _ in range(2):
        fn()
    ts = []
    for _ in range(reps):
        _flush()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2]


def copy_peak_gbs(reps):
    a = torch.empty(4 << 30, dtype=torch.uint8, device=DEV)
    b = torch.empty_like(a)
    t = eager_ms(lambda: b.copy_(a), reps)
    return 2 * a.numel() / t / 1e6


def cellout(card, peak, reps, emit):
    for NH, D in TAIL_H + WHOLE_H:
        H = NH * D
        g = torch.Generator(device="cpu").manual_seed(H)
        h = torch.randn(B, NH, S, D, generator=g).to(DEV, torch.bfloat16)
        x = torch.randn(B, S, H, generator=g).to(DEV, torch.float16)
        dy = torch.randn(B, S, H, generator=g).to(DEV, torch.float16)
        w, b, sk = ((1 + 0.1 * torch.randn(H, generator=g)).to(DEV) for _ in range(3))
        n = B * S * H
        t_fw = graph_ms(lambda: vil._cellout_fw_call(h, x, w, b, sk, 1e-6, torch.float16)[0], reps)
        t_bw = graph_ms(lambda: vil._cellout_bw_call(h, x, w, sk, dy, 1e-6, torch.float16, True), reps)
        hr, xr, wr, br, skr = (t.detach().requires_grad_(True) for t in (h, x, w, b, sk))

        def ref():
            with torch.autocast("cuda", dtype=torch.float16):
                y = F.group_norm(hr.to(torch.float16).transpose(1, 2).reshape(B * S, H), NH, wr, br, 1e-6)
                return y.view(B, S, H) + skr * xr

        t_rfw = eager_ms(ref, max(3, reps // 4))
        yr = ref()
        t_rbw = eager_ms(lambda: torch.autograd.grad(yr, (hr, xr, wr, br, skr), dy.to(yr.dtype), retain_graph=True),
                         max(3, reps // 4))
        del yr
        for kind, t, tr, nbytes in (("cellout_fw", t_fw, t_rfw, 6 * n), ("cellout_bw", t_bw, t_rbw, 10 * n)):
            emit(dict(kind=kind, H=H, NH=NH, D=D, tail=H % 128 != 0, B=B, S=S, ms=round(t, 4),
                      frac_of_copy_peak=round(nbytes / t / 1e6 / peak, 3), torch_ms=round(tr, 4),
                      speedup_vs_torch=round(tr / t, 2), card=card))
        del h, x, dy


def rmsnorm(card, peak, reps, emit):
    rows = B * S
    for C in RMS_NEW + RMS_SHIPPED:
        g = torch.Generator(device="cpu").manual_seed(C)
        x = torch.randn(rows, C, generator=g).to(DEV, torch.float16)
        dy = torch.randn(rows, C, generator=g).to(DEV, torch.float16)
        w = (1 + 0.1 * torch.randn(C, generator=g)).to(DEV)
        n = rows * C
        y, rstd = vil._rmsnorm_fw_call(x, w, 1e-6, torch.float16)
        t_fw = graph_ms(lambda: vil._rmsnorm_fw_call(x, w, 1e-6, torch.float16)[0], reps)
        t_bw = graph_ms(lambda: vil._rmsnorm_bw_call(x, w, rstd, dy, 1e-6, torch.float16), reps)
        xr, wr = x.detach().requires_grad_(True), w.detach().requires_grad_(True)

        def ref():
            with torch.autocast("cuda", dtype=torch.float16):
                return torch.rms_norm(xr, (C,), wr, 1e-6)

        t_rfw = eager_ms(ref, max(3, reps // 4))
        yr = ref()
        t_rbw = eager_ms(lambda: torch.autograd.grad(yr, (xr, wr), dy.to(yr.dtype), retain_graph=True), max(3, reps // 4))
        del yr
        for kind, t, tr, nbytes in (("rmsnorm_fw", t_fw, t_rfw, 4 * n), ("rmsnorm_bw", t_bw, t_rbw, 6 * n)):
            emit(dict(kind=kind, C=C, shipped_kernel=C in RMS_SHIPPED, rows=rows, ms=round(t, 4),
                      frac_of_copy_peak=round(nbytes / t / 1e6 / peak, 3), torch_ms=round(tr, 4),
                      speedup_vs_torch=round(tr / t, 2), card=card))
        del x, dy, y, rstd


def layer_step(card, reps, emit):
    from test_widths_gpu import _Layer

    torch.manual_seed(0)
    layer = _Layer(320, 128, False).to(DEV)
    layer.conv.seqlens = [80, 80]
    x = torch.randn(B, S, 320, device=DEV)
    dout = torch.randn(B, S, 320, device=DEV)

    def step():
        xi = x.detach().requires_grad_(True)
        layer.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.float16):
            y = layer(xi)
        y.backward(dout)

    res = {}
    for arm in ("unpatched", "patched"):
        if arm == "patched":
            assert pkg.patch_layers(layer) == 1
        res[arm] = eager_ms(step, reps)
    emit(dict(kind="layer_step", dim=320, inner=640, NH=5, D=128, B=B, S=S, unpatched_ms=round(res["unpatched"], 3),
              patched_ms=round(res["patched"], 3), speedup=round(res["unpatched"] / res["patched"], 2),
              timing="fwd+bwd, fp16 autocast, CUDA events around the eager step", card=card))


def main():
    global FLUSH
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "width_bench measures on a CUDA device"
    FLUSH = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
    card = _card()
    fh = open(args.out, "w") if args.out else None

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        if fh:
            fh.write(line + "\n")
            fh.flush()

    peak = copy_peak_gbs(args.reps)
    emit(dict(kind="copy_peak", gbs=round(peak, 1), bytes="read + write of 4 GiB", card=card))
    cellout(card, peak, args.reps, emit)
    torch.cuda.empty_cache()
    rmsnorm(card, peak, args.reps, emit)
    torch.cuda.empty_cache()
    layer_step(card, max(5, args.reps // 2), emit)


if __name__ == "__main__":
    main()
