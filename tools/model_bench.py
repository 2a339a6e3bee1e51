#!/usr/bin/env python
"""Model-level and kernel-level comparison against the reference's own CUDA path, on the GPU box.

Needs the unmodified reference staged by tools/stage_reference.sh under baseline/_ref/ (git-ignored; it is
the reference's ultralytics fork + mlstm_kernels, imported as they are).  Not part of bench.py / tests / smoke.

  python tools/model_bench.py kernel                      # BASELINE configs[1] microbench: reference Triton
                                                          # xl_chunk / xl_chunk_siging vs chunkwise--b200[_siging]
  python tools/model_bench.py train --yaml 640-base256.yaml --batch 32 [--backends triton,b200_siging,b200]
  python tools/model_bench.py infer --yaml 640-base384.yaml --batch 16
  torchrun --nproc-per-node N tools/model_bench.py train ...   # DDP (configs[3]): per-GPU batch, NCCL all-reduce

Backends: "triton" = the model exactly as the reference builds it (MatrixLSTMCell.gpu_backend =
chunkwise--triton_xl_chunk_siging, vision_lstm2.py:685-697); "b200_siging" / "b200" = the same model after
xlstm_yolo_clean_b200.patch_model().  Every line printed is JSON.
"""
import argparse
import json
import os
import statistics
import sys
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "baseline", "_ref")
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def _import_reference():
    if not os.path.isdir(os.path.join(REF, "mlstm_kernels")):
        raise SystemExit("baseline/_ref is missing: run `sh tools/stage_reference.sh <checkout of xlstm-yolo-clean>` first")
    sys.path.insert(0, REF)
    os.environ.setdefault("YOLO_CONFIG_DIR", "/tmp/yolo_cfg")
    for name in ("matplotlib", "matplotlib.pyplot"):  # hard import at ultralytics/utils/__init__.py:24
        try:
            __import__(name)
        except Exception:
            sys.modules[name] = types.ModuleType(name)
    if isinstance(sys.modules.get("matplotlib"), types.ModuleType) and not hasattr(sys.modules["matplotlib"], "pyplot"):
        sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]


def _events():
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def _time_cuda(fn, warmup, reps, flush=None):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        if flush is not None:
            flush.zero_()
        e0, e1 = _events()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return statistics.median(ts), min(ts)


# ------------------------------------------------------------------------------------------------
def run_kernel(args):
    """configs[1]: bf16 B=32 NH=4 S=1600 DH=64 chunk=64 fwd+bwd through the reference registry, every arm
    called the same way (autograd, contiguous inputs, eager launches, 256 MB L2 flush between reps as in
    mlstm_kernels/utils/benchmark/runtime.py:66-72)."""
    _import_reference()
    from mlstm_kernels.torch import get_mlstm_kernel

    import xlstm_yolo_clean_b200 as pkg
    from oracle import mlstm_oracle as O

    pkg.register()
    dev = torch.device("cuda", 0)
    B, NH, S, D = args.B, args.NH, args.S, args.D
    flops = 14 * 64 * D * (64 + D) * (S // 64) * B * NH
    inp = O.make_inputs(B, NH, S, D, D, seed=0, dtype=torch.float32)
    t = {k: v.to(torch.bfloat16).to(dev) for k, v in inp.items()}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ref64 = None
    for name in args.backends.split(","):
        full = {"triton": "chunkwise--triton_xl_chunk", "triton_siging": "chunkwise--triton_xl_chunk_siging",
                "triton_limit": "chunkwise--triton_limit_chunk", "native_custbw": "chunkwise--native_custbw", "native_autograd": "chunkwise--native_autograd",
                "b200": "chunkwise--b200", "b200_siging": "chunkwise--b200_siging"}[name]
        fn = get_mlstm_kernel(full)
        q, k, v, i, f = (t[n].clone().requires_grad_(True) for n in ("q", "k", "v", "i", "f"))
        kw = dict(chunk_size=64, eps=1e-6, autocast_kernel_dtype=torch.bfloat16)

        def fw():
            return fn(q=q, k=k, v=v, i=i, f=f, **kw)

        def fwbw():
            for x in (q, k, v, i, f):
                x.grad = None
            fw().backward(t["dh"])

        try:
            with torch.no_grad():
                fw_med, fw_min = _time_cuda(fw, 5, args.reps, flush)
            med, mn = _time_cuda(fwbw, 5, args.reps, flush)
        except Exception as e:  # a reference kernel that cannot run on this box is reported, not hidden
            sys.stderr.write(f"---- {name} failed ----\n{e}\n")
            print(json.dumps({"mode": "kernel", "backend": name, "error": str(e)[-600:]}))
            continue
        h = fw().detach().float()
        line = {"mode": "kernel", "backend": name, "kernel": full, "shape": [B, NH, S, D], "dtype": "bf16",
                "fwbw_ms_median": med, "fwbw_ms_min": mn, "fw_ms_median": fw_med, "fw_ms_min": fw_min,
                "tflops_median": flops / (med * 1e-3) / 1e12, "launch": "eager autograd call, L2 flushed"}
        if "siging" not in name:
            if ref64 is None:
                d = {k_: v_.to(torch.bfloat16).double() for k_, v_ in inp.items()}
                ref64 = O.chunkwise_fw(d["q"][:2], d["k"][:2], d["v"][:2], d["i"][:2], d["f"][:2])[0]
            line["h_rel_err_vs_fp64_oracle"] = O.rel_err(h[:2].cpu(), ref64)
        print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def _build_model(yaml_name, dev):
    from ultralytics.cfg import get_cfg
    from ultralytics.nn.tasks import DetectionModel

    torch.manual_seed(0)
    model = DetectionModel(os.path.join(REF, yaml_name), ch=3, nc=80, verbose=False)
    model.args = get_cfg()
    return model.to(dev)


def _batch(B, dev, seed):
    g = torch.Generator().manual_seed(seed)
    nb = 3  # boxes per image
    return {"img": torch.rand(B, 3, 640, 640, generator=g).to(dev),
            "cls": torch.randint(0, 80, (B * nb, 1), generator=g).float().to(dev),
            "bboxes": torch.cat([torch.rand(B * nb, 2, generator=g) * 0.5 + 0.25,
                                 torch.rand(B * nb, 2, generator=g) * 0.3 + 0.05], 1).to(dev),
            "batch_idx": torch.arange(B).repeat_interleave(nb).float().to(dev)}


def _set_backend(model, name):
    import xlstm_yolo_clean_b200 as pkg

    cells = [m for m in model.modules() if hasattr(m, "gpu_backend") and hasattr(m, "cpu_backend")]
    if name == "triton":
        return len(cells)
    if name in ("native_custbw", "native_autograd"):
        # the reference's own native-torch chunkwise kernels (its CPU default, vision_lstm2.py:670-682) run on CUDA
        from mlstm_kernels.torch.backend_module import mLSTMBackend, mLSTMBackendConfig
        for c in cells:
            c.gpu_backend = mLSTMBackend(mLSTMBackendConfig(
                chunkwise_kernel="chunkwise--" + name, sequence_kernel="native_sequence__native", step_kernel="native",
                mode="train_with_padding", return_last_states=False, chunk_size=64, eps=1e-6,
                autocast_kernel_dtype="bfloat16"))
        return len(cells)
    return pkg.patch_model(model, siging="siging" in name, fused="_fused" in name,
                           kernel_dtype="input" if "_fp16" in name else "bfloat16",
                           keep_activations="_keep" in name, graphs="_graphs" in name)


class _MlstmTimer:
    """CUDA-event timing of every mLSTMBackend.forward call (forward share of the step only)."""

    def __init__(self, model, check_finite=False):
        self.pairs, self.handles, self.check, self.bad = [], [], check_finite, []
        for m in model.modules():
            if hasattr(m, "gpu_backend") and hasattr(m, "cpu_backend"):
                self.handles.append(m.gpu_backend.register_forward_pre_hook(self._pre, with_kwargs=True))
                self.handles.append(m.gpu_backend.register_forward_hook(self._post))

    def _note(self, what, t):
        if not bool(torch.isfinite(t).all()):
            self.bad.append(f"{what} S={t.shape[2]} absmax={float(t.float().abs().nan_to_num(0, 0, 0).max()):.3g}")

    def _pre(self, mod, inp, kwargs):
        if self.check:
            for n in ("q", "k", "v", "i", "f"):
                t = kwargs[n]
                self._note("in:" + n, t)
                if t.requires_grad:
                    t.register_hook(lambda g, n=n: self._note("grad:" + n, g))
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.pairs.append([e, None])

    def _post(self, mod, inp, out):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.pairs[-1][1] = e
        if self.check:
            self._note("out:h", out)
            if out.requires_grad:
                out.register_hook(lambda g: self._note("grad:h", g))

    def total_ms(self):
        torch.cuda.synchronize()
        t = sum(a.elapsed_time(b) for a, b in self.pairs if b is not None)
        n = len(self.pairs)
        self.pairs = []
        return t, n

    def remove(self):
        for h in self.handles:
            h.remove()


def run_model(args, train):
    _import_reference()
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    for name in args.backends.split(","):
        model = _build_model(args.yaml, dev)
        cells = _set_backend(model, name)
        batch = _batch(args.batch, dev, seed=rank)
        err = None
        try:
            if train:
                res = _train_loop(model, batch, args, world, dev)
            else:
                res = _infer_loop(model, batch, args, dev)
        except Exception as e:
            sys.stderr.write(f"---- {name} failed ----\n{e}\n")
            err = str(e)[-600:]
            res = {}
        if world > 1:
            t = torch.tensor([res.get("ms_per_step", 0.0)], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            res["ms_per_step"] = float(t)
        if rank == 0:
            line = {"mode": "train" if train else "infer", "yaml": args.yaml, "backend": name, "cells": cells,
                    "n_gpus": world, "batch_per_gpu": args.batch, "steps": args.steps, **res}
            if err:
                line["error"] = err
            elif res.get("ms_per_step"):
                line["img_per_s"] = world * args.batch / (res["ms_per_step"] * 1e-3)
            print(json.dumps(line), flush=True)
        del model
        torch.cuda.empty_cache()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _train_loop(model, batch, args, world, dev):
    """One step = what BaseTrainer._do_train does per batch (engine/trainer.py:382-392,594-602): fp16 autocast
    forward + loss, scaled backward (DDP all-reduce), unscale, clip_grad_norm_(10), optimizer step."""
    from torch.nn.parallel import DistributedDataParallel as DDP

    model.train()
    # engine/trainer.py:277 uses find_unused_parameters=True; with torch 2.11 the reference's reentrant activation
    # checkpointing (vision_lstm2.py:1071-1078) then trips DDP's "marked ready twice" check, for the unmodified
    # reference model too, so the harness declares the graph static (the workaround the error message names).
    net = DDP(model, device_ids=[dev.index], find_unused_parameters=True, static_graph=True) if world > 1 else model
    opt = torch.optim.SGD(model.parameters(), lr=1e-3, momentum=0.937, nesterov=True)
    scaler = torch.amp.GradScaler("cuda", enabled=True)
    timer = _MlstmTimer(model, args.check_finite)
    losses = []

    def step():
        with torch.autocast("cuda", dtype=torch.float16):
            loss, items = net(batch)
            loss = loss.sum() * world
        scaler.scale(loss).backward()
        scaler.unscale_(opt)
        torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm=10.0)
        scaler.step(opt)
        scaler.update()
        opt.zero_grad(set_to_none=True)
        return loss

    for w in range(args.warmup):
        losses.append(float(step().detach()))
        if args.check_finite:
            sys.stderr.write(f"warmup step {w}: loss {losses[-1]} scale {scaler.get_scale()} non-finite: {timer.bad}\n")
            timer.bad = []
    timer.total_ms()
    if args.profile:
        from torch.profiler import ProfilerActivity, profile, record_function
        import xlstm_yolo_clean_b200.vil as _vil
        _cell = _vil.mlstm_cell_b200

        def _ranged_cell(*a, **kw):  # everything the fused cell launches in the forward (casts included) under one name
            with record_function("b200::mlstm_cell_forward"):
                return _cell(*a, **kw)

        _vil.mlstm_cell_b200 = _ranged_cell
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            step()
            torch.cuda.synchronize()
        sys.stderr.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=45, max_name_column_width=70) + "\n")
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.reset_peak_memory_stats()
    e0, e1 = _events()
    e0.record()
    for _ in range(args.steps):
        last = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    mlstm_ms, calls = timer.total_ms()
    timer.remove()
    return {"ms_per_step": ms, "first_loss": losses[0] if losses else None, "last_loss": float(last.detach()),
            "mlstm_forward_ms_per_step": mlstm_ms / args.steps, "mlstm_forward_calls_per_step": calls / args.steps,
            "peak_mem_gb": torch.cuda.max_memory_allocated() / 2**30,
            "step": "fp16 autocast fwd + loss, GradScaler backward, clip 10, SGD step; synthetic batch resident on device"}


def _infer_loop(model, batch, args, dev):
    model.eval()
    timer = _MlstmTimer(model)
    x = batch["img"]

    def step():
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
            return model(x)

    for _ in range(args.warmup):
        out = step()
    timer.total_ms()
    e0, e1 = _events()
    e0.record()
    for _ in range(args.steps):
        out = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    mlstm_ms, calls = timer.total_ms()
    timer.remove()
    y = out[0] if isinstance(out, (tuple, list)) else out
    y = y["one2one"] if isinstance(y, dict) else y
    return {"ms_per_step": ms, "mlstm_forward_ms_per_step": mlstm_ms / args.steps,
            "mlstm_forward_calls_per_step": calls / args.steps, "out_shape": list(y.shape) if hasattr(y, "shape") else None,
            "out_checksum": float(y.float().abs().mean()) if hasattr(y, "shape") else None,
            "peak_mem_gb": torch.cuda.max_memory_allocated() / 2**30}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("mode", choices=["kernel", "train", "infer"])
    ap.add_argument("--yaml", default="640-base256.yaml")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--backends", default=None)
    ap.add_argument("--check-finite", action="store_true")
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--B", type=int, default=32)
    ap.add_argument("--NH", type=int, default=4)
    ap.add_argument("--S", type=int, default=1600)
    ap.add_argument("--D", type=int, default=64)
    args = ap.parse_args()
    if args.backends is None:
        args.backends = "triton,triton_siging,b200,b200_siging" if args.mode == "kernel" else "triton,b200_siging,b200"
    if args.mode == "kernel":
        run_kernel(args)
    else:
        run_model(args, train=args.mode == "train")


if __name__ == "__main__":
    main()
