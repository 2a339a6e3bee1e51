"""Eager vs torch.compile vs torch.compile(mode="reduce-overhead") over the mlstm_b200 custom ops (needs a B200).

Workloads, forward + backward per step:
  * dropin_config2: ``mlstm_chunkwise__b200`` at BASELINE config 2 (bf16, B=32 NH=4 S=1600 DH=64, chunk 64);
  * layer_S<S>: a ViLLayer stand-in at the base256 call shapes (dim 256, inner 512, 8 heads of 64, B=32,
    S = 6400 / 1600 / 400 / 100): x + mlstm_branch_b200(RMSNorm(x)) under fp16 autocast, the bf16 kernels, the cell as
    the layer-layout mLSTM call + cell-output pass (one_launch="auto").

Per step it reports host time (wall clock of issuing the step, no synchronise inside) and device time (CUDA events
around the step), means over the timed steps after warm-up, with the card name and power limit read in the same run.

    python tools/compile_bench.py [--steps 30] [--warmup 10] [--out profiles/r05_compile_bench.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import xlstm_yolo_clean_b200 as pkg  # noqa: E402


class _Norm(torch.nn.Module):
    def __init__(self, H):
        super().__init__()
        self.weight = torch.nn.Parameter(0.1 * torch.randn(H))
        self.bias = torch.nn.Parameter(0.1 * torch.randn(H))
        self.eps = 1e-6

    @property
    def weight_proxy(self):
        return 1.0 + self.weight


class _Cell(torch.nn.Module):
    def __init__(self, H, NH):
        super().__init__()
        self.dim, self.num_heads, self.gate_soft_cap = H, NH, 15.0
        self.use_autocast, self.autocast_dtype = True, torch.float16
        self.ifgate = torch.nn.Linear(3 * H, 2 * NH)
        self.outnorm = _Norm(H)
        with torch.no_grad():
            self.ifgate.bias[:NH] = -2.0
            self.ifgate.bias[NH:] = torch.linspace(3.0, 6.0, NH)


class _Dir:
    name = "ROWWISE_FROM_TOP_LEFT"


class Layer(torch.nn.Module):
    """Attribute-compatible ViLLayer stand-in (proj_up, conv, qk_proj, v_proj, mlstm_cell, learnable_skip, proj_down)."""

    def __init__(self, dim=256, NH=8):
        super().__init__()
        inner = 2 * dim
        self.direction = _Dir()
        self.proj_up = torch.nn.Linear(dim, 2 * inner)
        self.conv = torch.nn.Conv2d(inner, inner, 3, padding=1, groups=inner)
        self.qk_proj = torch.nn.Linear(inner, 2 * inner)
        self.v_proj = torch.nn.Linear(inner, inner)
        self.mlstm_cell = _Cell(inner, NH)
        self.learnable_skip = torch.nn.Parameter(1.0 + 0.1 * torch.randn(inner))
        self.proj_down = torch.nn.Linear(inner, dim)
        self.norm = torch.nn.RMSNorm(dim, eps=1e-6)

    def forward(self, x):
        with torch.autocast("cuda", dtype=torch.float16):
            return x + pkg.mlstm_branch_b200(self, pkg.rms_norm_b200(x, self.norm.weight, 1e-6))


def _card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else torch.cuda.get_device_name()


def _time(step, steps, warmup, mark):
    for _ in range(warmup):
        mark()
        step()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    host = 0.0
    for a, b in ev:
        mark()
        a.record()
        t0 = time.perf_counter()
        step()
        host += time.perf_counter() - t0
        b.record()
    torch.cuda.synchronize()
    return host / steps * 1e3, sum(a.elapsed_time(b) for a, b in ev) / steps


def _dropin_step(fn):
    g = torch.Generator(device="cpu").manual_seed(0)
    B, NH, S, D = 32, 4, 1600, 64
    mk = lambda *s: torch.randn(*s, generator=g).to("cuda", torch.bfloat16).requires_grad_(True)  # noqa: E731
    ts = [mk(B, NH, S, D), mk(B, NH, S, D), mk(B, NH, S, D), mk(B, NH, S), mk(B, NH, S)]
    dh = torch.randn(B, NH, S, D, device="cuda", dtype=torch.bfloat16)

    def step():
        for t in ts:
            t.grad = None
        fn(*ts).backward(dh)

    return step


def _layer_step(fn, layer, S):
    x = torch.randn(32, S, 256, device="cuda", requires_grad=True)
    dout = torch.randn(32, S, 256, device="cuda")

    def step():
        x.grad = None
        layer.zero_grad(set_to_none=True)
        fn(x).backward(dout)

    return step


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("compile_bench.py needs a CUDA device (B200)")
    card = _card()
    dropin = lambda q, k, v, i, f: pkg.mlstm_chunkwise__b200(q, k, v, i, f, chunk_size=64, eps=1e-6)  # noqa: E731
    torch.manual_seed(0)
    layer = Layer().cuda()
    workloads = [("dropin_config2", lambda fn: _dropin_step(fn), dropin)]
    workloads += [(f"layer_S{S}", (lambda S: lambda fn: _layer_step(fn, layer, S))(S), layer) for S in (6400, 1600, 400, 100)]
    rows = []
    for name, make, fn in workloads:
        for mode in ("eager", "compile", "reduce-overhead"):
            torch._dynamo.reset()
            if mode == "eager":
                f, mark = fn, (lambda: None)
            else:
                f = torch.compile(fn, fullgraph=True, mode=None if mode == "compile" else "reduce-overhead")
                mark = torch.compiler.cudagraph_mark_step_begin if mode == "reduce-overhead" else (lambda: None)
            host_ms, dev_ms = _time(make(f), args.steps, args.warmup, mark)
            row = dict(workload=name, mode=mode, host_ms_per_step=round(host_ms, 4), device_ms_per_step=round(dev_ms, 4),
                       steps=args.steps, warmup=args.warmup, card=card, torch=torch.__version__)
            print(json.dumps(row), flush=True)
            rows.append(row)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.writelines(json.dumps(r) + "\n" for r in rows)


if __name__ == "__main__":
    main()
