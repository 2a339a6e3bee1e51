#!/usr/bin/env python
"""Benchmark of the hot path: mLSTM chunkwise fwd+bwd (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One "step" = one forward + one backward of the chunkwise mLSTM over one batch of synthetic
input: bf16, B=32 NH=4 S=1600 DH=64 chunk=64 per GPU (weak scaling: every rank runs the same
per-GPU workload on its own data; the op has no cross-sample term, so there is no data-path
collective -- SURVEY.md §8e).  Prints ONE JSON line (rank 0).

--dump-outputs DIR writes what the last timed step returned (rank 0) as DIR/<name>.npy in float32, so that two
builds can be compared output for output: the inputs are seeded, identical from run to run.

Metric: algorithmic TFLOP/s = 14*L*d*(L+d) FLOP per chunk (SURVEY.md §8d) x chunks / time.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

CFG = dict(B=32, NH=4, S=1600, DK=64, DV=64, L=64)
WORKLOAD = "mlstm_chunkwise_fwbw bf16 B=32 NH=4 S=1600 DH=64 chunk=64 (BASELINE configs[1])"
METRIC = "mLSTM chunkwise fwd+bwd TFLOP/s (algorithmic, 14*L*d*(L+d) per chunk)"
N_SETS = 4  # rotating input sets: ~105 MB of inputs + ~105 MB of outputs per step >> 126 MB L2 over a rotation
DUMP_BYTES = 60_000_000  # --dump-outputs stays under 64 MB: one step's outputs are ~213 MB in float32


def flops_and_bytes(c, itemsize=2):
    """Algorithmic FLOPs / bytes per step per GPU (SURVEY.md §8d)."""
    nc = c["S"] // c["L"]
    bh = c["B"] * c["NH"]
    fwd = 4 * c["L"] * c["DK"] * c["DV"] + 2 * c["L"] ** 2 * (c["DK"] + c["DV"])
    bwd = 10 * c["L"] * c["DK"] * c["DV"] + 2 * c["L"] ** 2 * (3 * c["DK"] + 2 * c["DV"])
    tok = bh * c["S"]
    qk, v = tok * c["DK"] * itemsize, tok * c["DV"] * itemsize
    gate, vec32 = tok * itemsize, tok * 4
    fw_bytes = 2 * qk + v + 2 * gate + v + 2 * vec32  # read q,k,v,i,f; write h,n_out,m_out
    bw_bytes = 2 * qk + v + v + 2 * gate + 2 * vec32 + 2 * qk + v + 2 * gate  # read q,k,v,dh,i,f,n,m; write dq,dk,dv,di,df
    return bh * nc * fwd, bh * nc * bwd, fw_bytes, bw_bytes


def dump_outputs(out_dir, outs, seed=0):
    """Write each (B, NH, ...) output as out_dir/<name>.npy in float32, its (batch, head) rows flattened into one
    leading axis.  Where all rows do not fit DUMP_BYTES, every array keeps the same fixed, seeded subset of rows
    (ascending (batch, head) order), so that row r of every file belongs to the same (batch, head)."""
    import numpy as np

    rows = {name: t.detach().flatten(0, 1) for name, t in outs.items()}
    n_rows = next(iter(rows.values())).shape[0]
    row_bytes = sum(t[0].numel() * 4 for t in rows.values())
    keep = min(n_rows, DUMP_BYTES // row_bytes)
    idx = torch.randperm(n_rows, generator=torch.Generator().manual_seed(seed))[:keep].sort().values
    os.makedirs(out_dir, exist_ok=True)
    for name, t in rows.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t[idx.to(t.device)].float().cpu().numpy())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler:
    """SM clock / throttle reasons sampled through NVML DURING the timed region (the nvidia-smi
    subprocess of the profiling recipe stalls kernel launches of a sub-millisecond step, so the
    same counters are read in-process)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index, self.sm, self.bits, self.max_mhz = index, [], 0, None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml

            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # pragma: no cover
            self.nv, self.err = None, repr(e)

    def _sample(self):
        self.sm.append(float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
        try:
            self.bits |= int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
        except Exception:
            self.bits |= int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))

    def _loop(self):
        while not self._stop.is_set():
            self._sample()
            time.sleep(0.002)

    def start(self):
        if self.nv is None:
            return
        self._thr = threading.Thread(target=self._loop, daemon=True)
        self._thr.start()

    def stop(self):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "?")]}
        self._sample()
        self._stop.set()
        if self._thr:
            self._thr.join()
        reasons = sorted(n for b, n in self.REASONS.items() if self.bits & b)
        return {"sm_mhz": statistics.median(self.sm), "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(self.sm)}


def _oracle_step(c, seed=0):
    """Inputs + one fp32 fwd+bwd step of the reference's native-torch formulation (oracle port) on the host cores."""
    from oracle import mlstm_oracle as O

    inp = O.make_inputs(c["B"], c["NH"], c["S"], c["DK"], c["DV"], seed=seed, dtype=torch.float32)

    def step():
        # the reference's custbw path: forward, then the hand-written backward with the saved n / m vectors
        # (native/fwbw.py:34-171); no autograd graph is involved in either, grad mode is left on as in training
        return O.fwbw(inp["q"], inp["k"], inp["v"], inp["i"], inp["f"], inp["dh"], chunk_size=c["L"])

    return step


def cpu_baseline(sample_b=8, reps=2):
    """Oracle port (native-torch formulation) in fp32 on the host cores, on a bounded sample (rank 0, N = 1 only)."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    c = dict(CFG, B=sample_b)
    step = _oracle_step(c)
    best = float("inf")
    for r in range(reps + 1):
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        if r:
            best = min(best, dt)
    ff, fb, _, _ = flops_and_bytes(c, 4)
    return {"value": (ff + fb) / best / 1e12, "unit": "TFLOP/s", "cores": cores, "kind": "port",
            "sample": f"fp32 fwd+bwd of B={sample_b} (of 32) NH=4 S=1600 DH=64 chunk=64, best of {reps}, {best * 1e3:.1f} ms",
            "seconds": best}


def run_reference(args, rank):
    """--impl reference: the reference's CPU formulation (oracle port; the Python reference cannot travel to the GPU
    box) on all host cores, on the SAME configuration as the B200 arm: every step is the full B=32 fwd+bwd."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    c = dict(CFG)
    step = _oracle_step(c)
    times = []
    for s in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        step()
        if s >= args.warmup:
            times.append(time.perf_counter() - t0)
    ff, fb, _, _ = flops_and_bytes(c, 4)
    dt = sum(times) / len(times)
    val = (ff + fb) / dt / 1e12
    sample = "each step = the full configuration: fp32 fwd+bwd of B=32 NH=4 S=1600 DH=64 chunk=64 on the host cores"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "TFLOP/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "per_gpu": True, "sample": sample, "same_config": True},
        "cpu_baseline": {"value": val, "unit": "TFLOP/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# --------------------------------------------------------------------------------------------------------------
# The calls a YOLO-ViL step makes (SURVEY.md section 3.1): 10 block pairs x 2 directions per forward pass, at four stage
# resolutions; in training the two S = 6400 pairs are activation-checkpointed, so a step runs 24 forwards + 20
# backwards.  S = 400 / 100 are what the fused layer path hands to the kernels (ragged last 128-token tile handled
# in-kernel); the reference's pad wrapper would make them 448 / 128.
MODEL_CALLS = {
    "config3 640-base192 train, 64 img": dict(B=64, NH=12, D=32, train=True),
    "config4 640-base256 train, 32 img per GPU": dict(B=32, NH=8, D=64, train=True),
    "config5 640-base384 inference, 16 img per GPU": dict(B=16, NH=6, D=128, train=False),
}
STAGE_CALLS = ((6400, 4), (1600, 6), (400, 6), (100, 4))  # (S, calls per forward pass)


def call_bytes(B, NH, S, D, itemsize=2):
    tok = B * NH * S
    fw = tok * (4 * D * itemsize + 2 * itemsize + 8)
    bw = tok * (7 * D * itemsize + 4 * itemsize + 8)
    return fw, bw


def _graph_period(fn, reps, dev):
    """Device time per call: `reps` back-to-back calls captured in one CUDA graph (launch latency amortised)."""
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


def model_calls_block(pkg, dev, hbm_peak, flush):
    """Every mLSTM call shape of BASELINE configs 3 / 4 / 5, timed on its own: device time of the kernels (graph of
    back-to-back launches; the working set of the S >= 1600 calls exceeds the 126 MB L2) with the fraction of the measured
    HBM peak their algorithmic bytes reach, and the wall time of one eager call through the registered drop-in
    (autograd fwd+bwd, or the forward under no_grad for the inference config) with the L2 flushed between calls."""
    out = {}
    for name, c in MODEL_CALLS.items():
        B, NH, D, train = c["B"], c["NH"], c["D"], c["train"]
        rows, step_dev, step_eager = [], 0.0, 0.0
        for S, n_fw in STAGE_CALLS:
            g = torch.Generator(device=dev).manual_seed(S + D)
            t = {k: (0.3 * torch.randn(B, NH, S, D, generator=g, device=dev)).to(torch.bfloat16) for k in ("q", "k", "v", "dh")}
            t["i"] = torch.full((B, NH, S), -8.73, device=dev).to(torch.bfloat16)
            t["f"] = (3.0 + 3.0 * torch.rand(B, NH, S, generator=g, device=dev)).to(torch.bfloat16)
            L = 64 if S % 64 == 0 else 4
            reps = 4 if S >= 1600 else 16
            saved = pkg.mlstm_chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=L, save_states=train)
            fw_ms = _graph_period(lambda: pkg.mlstm_chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=L,
                                                                save_states=train), reps, dev)
            fwb, bwb = call_bytes(B, NH, S, D)
            row = {"S": S, "heads": B * NH, "d": D, "calls_fw": n_fw + (4 if (train and S == 6400) else 0), "fw_us": fw_ms * 1e3,
                   "fw_gbs": fwb / fw_ms / 1e6, "fw_frac": fwb / fw_ms / 1e6 / hbm_peak}
            if train:
                bw_ms = _graph_period(lambda: pkg.mlstm_chunkwise_bw(t["q"], t["k"], t["v"], t["i"], t["f"], saved[1], saved[2],
                                                                    t["dh"], chunk_size=L, c_states=saved[4]), reps, dev)
                row.update(calls_bw=n_fw, bw_us=bw_ms * 1e3, bw_gbs=bwb / bw_ms / 1e6, bw_frac=bwb / bw_ms / 1e6 / hbm_peak)
            # eager drop-in call (what the model pays per call when it is not launch-bound elsewhere)
            leaves = {k: t[k].detach().requires_grad_(train) for k in ("q", "k", "v", "i", "f")}

            def eager():
                if train:
                    h = pkg.mlstm_chunkwise__b200(**leaves, chunk_size=L)
                    h.backward(t["dh"])
                    for x in leaves.values():
                        x.grad = None
                else:
                    with torch.no_grad():
                        pkg.mlstm_chunkwise__b200(**leaves, chunk_size=L)

            for _ in range(3):
                eager()
            ts = []
            for _ in range(5):
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                eager()
                b.record()
                torch.cuda.synchronize()
                ts.append(a.elapsed_time(b))
            row["eager_dropin_us"] = statistics.median(ts) * 1e3
            rows.append(row)
            step_dev += row["calls_fw"] * row["fw_us"] + row.get("calls_bw", 0) * row.get("bw_us", 0.0)
            del t, saved, leaves
            torch.cuda.empty_cache()
        out[name] = {"calls": rows, "mlstm_device_ms_per_step": step_dev / 1e3}
    return out


def bind_numa_near_gpu(local_rank):
    """Pin this rank's threads and future host allocations (the pinned e2e buffers) to the NUMA node its GPU hangs off:
    with all ranks on node 0 the 8-GPU e2e run was bound by one socket's memory / PCIe root (round-1 VERDICT).  Best
    effort (sysfs + the raw set_mempolicy syscall; no libnuma in the image); returns what it did."""
    try:
        import ctypes

        import pynvml

        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[local_rank]) if vis and vis.split(",")[local_rank].isdigit() else local_rank
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(phys)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        bus = bus[-12:] if len(bus) > 12 else bus  # sysfs uses a 4-digit PCI domain
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return {"numa_node": None, "note": "single NUMA node / not reported"}
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.extend(range(int(lo), int(hi or lo) + 1))
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
        mask = ctypes.c_ulong(1 << node)
        rc = ctypes.CDLL(None, use_errno=True).syscall(238, 1, ctypes.byref(mask), 64)  # set_mempolicy(MPOL_PREFERRED)
        return {"numa_node": node, "cpus": len(allowed), "mempolicy_rc": int(rc)}
    except Exception as e:  # pragma: no cover
        return {"numa_node": None, "note": repr(e)[:120]}


def ddp_proxy_block(pkg, dist, dev, world, flush):
    """N > 1: the data-parallel pattern of BASELINE config 4 around the hot path -- per rank the mLSTM call sequence of
    one 640-base256 training step at 32 img per GPU (24 forwards + 20 backwards), and the gradient all-reduce DDP issues
    for that model (187 MB fp32, 25 MB buckets: engine/trainer.py:277, torch DDP defaults) over NCCL, launched bucket by
    bucket while the backward calls run.  Reports the three times (calls alone, all-reduce alone, overlapped) and which
    one bounds the step: the op itself has no collective, this is the one around it."""
    c = MODEL_CALLS["config4 640-base256 train, 32 img per GPU"]
    B, NH, D = c["B"], c["NH"], c["D"]
    ts = {}
    for S, _ in STAGE_CALLS:
        g = torch.Generator(device=dev).manual_seed(S)
        t = {k: (0.3 * torch.randn(B, NH, S, D, generator=g, device=dev)).to(torch.bfloat16) for k in ("q", "k", "v", "dh")}
        t["i"] = torch.full((B, NH, S), -8.73, device=dev).to(torch.bfloat16)
        t["f"] = (3.0 + 3.0 * torch.rand(B, NH, S, generator=g, device=dev)).to(torch.bfloat16)
        t["L"] = 64 if S % 64 == 0 else 4
        ts[S] = t
    n_bucket, bucket_elems = 8, (187 << 20) // 4 // 8
    buckets = [torch.ones(bucket_elems, device=dev) for _ in range(n_bucket)]
    comm = torch.cuda.Stream(dev)

    def forward_calls():
        saved = {}
        for S, n in STAGE_CALLS:
            t = ts[S]
            for _ in range(n):
                saved[S] = pkg.mlstm_chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=t["L"])
        return saved

    def backward_calls(saved, with_comm):
        k = 0
        for S, n in reversed(STAGE_CALLS):
            t = ts[S]
            for j in range(n):
                if S == 6400:  # checkpointed block pairs: the forward is recomputed inside the backward
                    saved[S] = pkg.mlstm_chunkwise_fw(t["q"], t["k"], t["v"], t["i"], t["f"], chunk_size=t["L"])
                pkg.mlstm_chunkwise_bw(t["q"], t["k"], t["v"], t["i"], t["f"], saved[S][1], saved[S][2], t["dh"],
                                       chunk_size=t["L"], c_states=saved[S][4])
                if with_comm and (j % 3 == 2 or j == n - 1) and k < n_bucket:  # a bucket fills every few layers
                    comm.wait_stream(torch.cuda.current_stream(dev))
                    with torch.cuda.stream(comm):
                        dist.all_reduce(buckets[k])
                    k += 1
        if with_comm:
            with torch.cuda.stream(comm):
                for kk in range(k, n_bucket):
                    dist.all_reduce(buckets[kk])
            torch.cuda.current_stream(dev).wait_stream(comm)

    def timed(fn, reps=3):
        best = float("inf")
        for _ in range(reps):
            flush.zero_()
            torch.cuda.synchronize()
            dist.barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            best = min(best, a.elapsed_time(b))
        return best

    def calls_only():
        backward_calls(forward_calls(), False)

    def comm_only():
        for x in buckets:
            dist.all_reduce(x)

    def overlapped():
        backward_calls(forward_calls(), True)

    for fn in (calls_only, comm_only, overlapped):
        fn()
    torch.cuda.synchronize()
    from xlstm_yolo_clean_b200 import replicas

    t_calls = replicas.max_over_ranks(timed(calls_only), dev)
    t_comm = replicas.max_over_ranks(timed(comm_only), dev)
    t_both = replicas.max_over_ranks(timed(overlapped), dev)
    bus_gbs = 2 * (world - 1) / world * (187 << 20) / (t_comm * 1e-3) / 1e9
    limiter = "mLSTM calls (the all-reduce hides behind them)" if t_both < 1.1 * t_calls else (
        "gradient all-reduce" if t_comm > t_calls else "launch / stream serialisation of calls and all-reduce")
    return {"workload": "640-base256 step per rank: 24 fw + 20 bw mLSTM calls (32 img per GPU) + all-reduce of 187 MB fp32 in 8 buckets",
            "mlstm_calls_ms": t_calls, "allreduce_ms": t_comm, "overlapped_ms": t_both,
            "allreduce_bus_gbs": bus_gbs, "overlap_efficiency": max(t_calls, t_comm) / t_both, "limiter": limiter,
            "images_per_s_bound_by_this_path": world * B / (t_both * 1e-3)}


def model_train_block(pkg, dist, dev, rank, world, steps=3, warmup=2):
    """The second half of BASELINE.json's metric -- 640-base256 training img/s -- through the reference's OWN model:
    the unmodified YOLO-ViL DetectionModel staged under baseline/_ref (git-ignored; it travels to the GPU box with the
    snapshot), patched with patch_model(fused=True), 32 synthetic 640x640 images per GPU, fp16 AMP, SGD step, DDP with
    NCCL gradient all-reduce when N > 1 (engine/trainer.py:221-232, 277, 382-392).  At N = 1 the same model with the
    reference's native-torch kernels on the GPU is timed beside it.  Absent reference -> {"unavailable": ...}."""
    import contextlib
    import types

    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import model_bench as MB

        if not os.path.isdir(os.path.join(MB.REF, "mlstm_kernels")):
            return {"unavailable": "baseline/_ref is not staged (tools/stage_reference.sh)"}
        out = {"model": "640-base256.yaml (DetectionModel, 80 classes)", "img_per_gpu": 32, "amp": "fp16", "n_gpus": world,
               "step": "autocast fwd + loss, GradScaler backward (DDP all-reduce at N > 1), clip 10, SGD step; synthetic batch"}
        args = types.SimpleNamespace(yaml="640-base256.yaml", batch=32, steps=steps, warmup=warmup, check_finite=False, profile=False)
        with contextlib.redirect_stdout(sys.stderr):
            MB._import_reference()
            for name in (["b200_fused"] + (["b200_fused_graphs", "b200_fused_graphs_keep_activations",
                                              "reference_native_custbw_on_gpu"] if world == 1 else [])):
                model = MB._build_model(args.yaml, dev)
                if name.startswith("b200_fused"):
                    # siging derived from the model's own CUDA backend; "_graphs": the layers' training forward /
                    # backward replay as CUDA graphs (single-process only, vil._Graphed); "_keep_activations": the
                    # S = 6400 block pairs are not re-run inside the backward (the reference checkpoints them to fit
                    # 40-80 GB parts; the step peaks at ~40 of the B200's 180 GB without)
                    pkg.patch_model(model, fused=True, graphs="_graphs" in name, keep_activations="_keep_activations" in name)
                else:
                    MB._set_backend(model, "native_custbw")
                res = MB._train_loop(model, MB._batch(32, dev, seed=rank), args, world, dev)
                ms = res["ms_per_step"]
                if world > 1:
                    t = torch.tensor([ms], device=dev)
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                    ms = float(t)
                out[name] = {"ms_per_step": ms, "img_per_s": world * 32 / (ms * 1e-3), "peak_mem_gb": res["peak_mem_gb"]}
                del model
                torch.cuda.empty_cache()
        return out
    except Exception as e:  # the block must never break the JSON line
        return {"error": repr(e)[:300]}


def model_infer_block(pkg, dev):
    """BASELINE configs 1 and 5 through the reference's own model (N = 1 only): 640-base192 single-image forward latency
    and 640-base384 forward throughput at 16 images per GPU, fp16 autocast, no_grad, with patch_model(fused=True) and with
    the layers' forward additionally replayed as CUDA graphs (graphs=True)."""
    import contextlib
    import types

    sys.path.insert(0, os.path.join(ROOT, "tools"))
    try:
        import model_bench as MB

        if not os.path.isdir(os.path.join(MB.REF, "mlstm_kernels")):
            return {"unavailable": "baseline/_ref is not staged (tools/stage_reference.sh)"}
        out = {"amp": "fp16", "step": "model(x) under no_grad + autocast, synthetic images resident on the device"}
        with contextlib.redirect_stdout(sys.stderr):
            MB._import_reference()
            for cfg, yaml_name, batch, steps in (("config1_base192_b1", "640-base192.yaml", 1, 20), ("config5_base384_b16", "640-base384.yaml", 16, 8)):
                args = types.SimpleNamespace(yaml=yaml_name, batch=batch, steps=steps, warmup=4)
                out[cfg] = {}
                for name, graphs in (("b200_fused", False), ("b200_fused_graphs", True)):
                    model = MB._build_model(yaml_name, dev)
                    pkg.patch_model(model, fused=True, graphs=graphs)
                    res = MB._infer_loop(model, MB._batch(batch, dev, seed=0), args, dev)
                    out[cfg][name] = {"ms_per_step": res["ms_per_step"], "img_per_s": batch / (res["ms_per_step"] * 1e-3),
                                      "out_checksum": res["out_checksum"]}
                    del model
                    torch.cuda.empty_cache()
        return out
    except Exception as e:  # the block must never break the JSON line
        return {"error": repr(e)[:300]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--kernel-impl", default="auto", choices=["auto", "exact", "tensor"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-model-calls", action="store_true")
    ap.add_argument("--no-model-train", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step (h, n_out, m_out, dq, dk, dv, di, df) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch.distributed as dist

    import __graft_entry__ as G

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the B200 backend has no CPU fallback")
    if local_rank == 0 and not os.path.exists(os.path.join(ROOT, "xlstm_yolo_clean_b200", "lib", "libmlstm_b200.so")):
        G.build()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL writes its version banner / debug lines to STDOUT when NCCL_DEBUG is set in the environment (the GPU
        # boxes export it); stdout carries the one JSON line only, so NCCL's output goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
            os.environ.pop("NCCL_DEBUG")
        dist.init_process_group("nccl", device_id=dev)
        dist.barrier()
    import xlstm_yolo_clean_b200 as pkg
    from oracle import mlstm_oracle as O

    pkg.set_default_impl(args.kernel_impl)
    c = CFG
    dt = torch.bfloat16
    sets = []
    for r in range(N_SETS):
        inp = O.make_inputs(c["B"], c["NH"], c["S"], c["DK"], c["DV"], seed=1000 * rank + r, dtype=torch.float32)
        sets.append({k: v.to(dt).to(dev) for k, v in inp.items()})
    ff, fb, fw_bytes, bw_bytes = flops_and_bytes(c)

    def fw_only(s):
        return pkg.mlstm_chunkwise_fw(s["q"], s["k"], s["v"], s["i"], s["f"], chunk_size=c["L"])

    def bw_only(s, saved):
        h, n_out, m_out, _, cst = saved
        return pkg.mlstm_chunkwise_bw(s["q"], s["k"], s["v"], s["i"], s["f"], n_out, m_out, s["dh"], chunk_size=c["L"],
                                      c_states=cst)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # eager warm-up (also counts the kernels one step launches)
    launches_per_step = 0
    for w in range(max(args.warmup, 3)):
        saved = fw_only(sets[w % N_SETS])
        n1 = pkg.last_launch_count()
        bw_only(sets[w % N_SETS], saved)
        launches_per_step = n1 + pkg.last_launch_count()
    torch.cuda.synchronize()

    # One CUDA graph per rotating input set: the step is two ~100 us kernels, so eager Python/ctypes
    # launch gaps would dominate.  Outputs live in the graphs' private pools.
    graphs, fw_graphs, bw_graphs, keep = [], [], [], []
    multi_out, single_out = [], []  # (forward, backward) results of the timed graphs, per input set
    side = torch.cuda.Stream()
    REP = 4  # launches per input set in the per-kernel graphs below
    with torch.cuda.stream(side):
        # N_SETS consecutive steps (one per rotating input set) in ONE graph: the ~6 us of graph-launch latency a
        # 90 us step would otherwise pay per replay is paid once per N_SETS steps
        g_multi = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g_multi, stream=side):
            for r in range(N_SETS):
                saved = fw_only(sets[r])
                multi_out.append((saved, bw_only(sets[r], saved)))
        # per-kernel graphs: REP * N_SETS back-to-back launches of ONE kernel over the rotating sets, so that the
        # roofline's per-launch duration is the kernel period, not kernel + graph launch + event overhead
        saved_all = [fw_only(sets[r]) for r in range(N_SETS)]
        g_fw_multi = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g_fw_multi, stream=side):
            for k in range(REP * N_SETS):
                keep.append(fw_only(sets[k % N_SETS]))
        g_bw_multi = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g_bw_multi, stream=side):
            for k in range(REP * N_SETS):
                keep.append(bw_only(sets[k % N_SETS], saved_all[k % N_SETS]))
        for r in range(N_SETS):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side):
                saved = fw_only(sets[r])
                out = bw_only(sets[r], saved)
            graphs.append(g)
            single_out.append((saved, out))
            gf = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gf, stream=side):
                saved_f = fw_only(sets[r])
            gb = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gb, stream=side):
                out_b = bw_only(sets[r], saved_f)
            fw_graphs.append(gf)
            bw_graphs.append(gb)
            keep.append((saved_f, out_b))
    torch.cuda.synchronize()

    # ---- device-resident throughput ("value") -------------------------------------------------
    for w in range(args.warmup):
        graphs[w % N_SETS].replay()
    g_multi.replay()
    sampler = ClockSampler(local_rank)
    sync_all()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(args.steps // N_SETS):  # EXACTLY args.steps steps: N_SETS per replay, the remainder one by one
        g_multi.replay()
    for k in range(args.steps % N_SETS):
        graphs[k].replay()
    e1.record()
    sync_all()
    clocks = sampler.stop() if rank == 0 else None
    launches = launches_per_step * args.steps
    from xlstm_yolo_clean_b200 import replicas

    ms_step = replicas.max_over_ranks(e0.elapsed_time(e1), dev) / args.steps  # slowest rank
    value = replicas.sum_over_ranks(ff + fb, dev) / (ms_step * 1e-3) / 1e12    # all ranks' work over that time
    if args.dump_outputs and rank == 0:
        rem = args.steps % N_SETS  # the last timed step is graphs[rem - 1], or the last set of g_multi
        (h, n_out, m_out, _, _), (dq, dk, dv, di, df, _) = single_out[rem - 1] if rem else multi_out[-1]
        dump_outputs(args.dump_outputs, dict(h=h, n_out=n_out, m_out=m_out, dq=dq, dk=dk, dv=dv, di=di, df=df))

    # ---- per-kernel timing for the roofline: CUDA events on the launching stream, one kernel per graph
    fw_ms, bw_ms = [], []
    for k in range(max(8, min(args.steps, 40))):
        r = k % N_SETS
        a, b_, c_ = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        a.record()
        fw_graphs[r].replay()
        b_.record()
        bw_graphs[r].replay()
        c_.record()
        torch.cuda.synchronize()
        fw_ms.append(a.elapsed_time(b_))
        bw_ms.append(b_.elapsed_time(c_))
    fw_single, bw_single = statistics.median(fw_ms), statistics.median(bw_ms)
    fw_ms, bw_ms = [], []
    for k in range(10):
        a, b_, c_ = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        a.record()
        g_fw_multi.replay()
        b_.record()
        g_bw_multi.replay()
        c_.record()
        torch.cuda.synchronize()
        fw_ms.append(a.elapsed_time(b_) / (REP * N_SETS))
        bw_ms.append(b_.elapsed_time(c_) / (REP * N_SETS))
    fw_t, bw_t = statistics.median(fw_ms), statistics.median(bw_ms)
    hbm_peak, tf_peak, peak_kind = peaks()
    dom = ("bw", bw_bytes, bw_t, "tc_bw") if bw_t >= fw_t else ("fw", fw_bytes, fw_t, "tc_fw")
    traffic = None  # DRAM bytes per launch of the dominant kernel from the committed ncu capture (same workload)
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))[dom[3]]
        traffic = tj["dram_read_bytes"] + tj["dram_write_bytes"] if args.kernel_impl == "auto" else None
    except Exception:
        pass
    roof = {"bound": "hbm", "kernel": f"{dom[3]} (mlstm_b200_chunkwise_{dom[0]}, one launch per call)",
            "achieved": dom[1] / (dom[2] * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
            "frac": dom[1] / (dom[2] * 1e-3) / 1e9 / hbm_peak, "traffic": traffic,
            "traffic_source": "static: committed ncu --set full capture of the same command (profiles/r02_traffic.json), not measured in this run" if traffic else None,
            "peak_kind": peak_kind,
            "algorithmic_bytes": dom[1], "fw_ms": fw_t, "bw_ms": bw_t,
            # the saved per-tile states are extra traffic the kernels really move (written by fw, read by bw); they are NOT
            # counted in the algorithmic bytes above (SURVEY.md section 8d: "no state materialisation")
            "c_states_bytes_each_way": c["B"] * c["NH"] * ((c["S"] + 127) // 128) * c["DK"] * c["DV"] * 2,
            "timing": f"CUDA events around a graph of {REP * N_SETS} back-to-back launches of the one kernel over the rotating input sets, / {REP * N_SETS}",
            "fw_ms_single_launch_graph": fw_single, "bw_ms_single_launch_graph": bw_single,
            "fw_gbs": fw_bytes / (fw_t * 1e-3) / 1e9, "bw_gbs": bw_bytes / (bw_t * 1e-3) / 1e9,
            "fw_frac": fw_bytes / (fw_t * 1e-3) / 1e9 / hbm_peak, "bw_frac": bw_bytes / (bw_t * 1e-3) / 1e9 / hbm_peak,
            "tflops_frac_of_bf16_peak": (ff + fb) / ((fw_t + bw_t) * 1e-3) / 1e12 / tf_peak}

    # ---- the same step through the registered drop-in (autograd.Function, eager launches): what a model pays --------
    leaves = [{k: st[k].detach().requires_grad_(True) for k in ("q", "k", "v", "i", "f")} for st in sets]

    def dropin_step(r):
        lv = leaves[r]
        h = pkg.mlstm_chunkwise__b200(**lv, chunk_size=c["L"])
        h.backward(sets[r]["dh"])
        for x in lv.values():
            x.grad = None

    for w in range(8):
        dropin_step(w % N_SETS)
    torch.cuda.synchronize()
    d_steps = max(8, min(args.steps, 100))
    e0.record()
    for k in range(d_steps):
        dropin_step(k % N_SETS)
    e1.record()
    sync_all()
    dropin_ms = replicas.max_over_ranks(e0.elapsed_time(e1), dev) / d_steps
    t0 = time.perf_counter()
    for k in range(200):
        dropin_step(k % N_SETS)
    host_us = (time.perf_counter() - t0) / 200 * 1e6  # (the GPU queue may throttle this when the host is faster)
    torch.cuda.synchronize()
    dropin = {"api": "mlstm_chunkwise__b200 (registered drop-in) + autograd backward, eager launches, rotating input sets",
              "ms_per_step": dropin_ms, "value": replicas.sum_over_ranks(ff + fb, dev) / (dropin_ms * 1e-3) / 1e12,
              "unit": "TFLOP/s", "host_us_per_step": host_us}
    # the same autograd step captured in a CUDA graph (forward AND backward through the autograd.Function): the
    # launch-bound part of the eager number is PyTorch's autograd engine, not the C-ABI call
    try:
        gd = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            for r in range(N_SETS):
                dropin_step(r)
            with torch.cuda.graph(gd, stream=side):
                for r in range(N_SETS):
                    dropin_step(r)
        torch.cuda.synchronize()
        gd.replay()
        sync_all()
        e0.record()
        for _ in range(max(2, d_steps // N_SETS)):
            gd.replay()
        e1.record()
        sync_all()
        g_ms = replicas.max_over_ranks(e0.elapsed_time(e1), dev) / (max(2, d_steps // N_SETS) * N_SETS)
        dropin["graph_captured_ms_per_step"] = g_ms
        dropin["graph_captured_value"] = replicas.sum_over_ranks(ff + fb, dev) / (g_ms * 1e-3) / 1e12
    except Exception as e:  # pragma: no cover
        dropin["graph_capture_error"] = repr(e)[:200]

    # ---- end to end through the public host-buffer API: pinned host tensors in, pinned host tensors out,
    #      H2D / kernels / D2H pipelined over batch slices (xlstm_yolo_clean_b200.HostFwBw) -----------
    numa = bind_numa_near_gpu(local_rank)
    host = {k: v.cpu().pin_memory() for k, v in sets[0].items()}
    pipe = pkg.HostFwBw(c["B"], c["NH"], c["S"], c["DK"], c["DV"], dtype=dt, device=dev, n_slices=1, lanes=2, chunk_size=c["L"])
    host_out = pkg.HostFwBw.alloc_host(c["B"], c["NH"], c["S"], c["DK"], c["DV"], dtype=dt)
    h2d, d2h = pipe.h2d_bytes, pipe.d2h_bytes
    for _ in range(4):
        pipe.run(host, host_out)
    pipe.flush()
    sync_all()
    e_steps = max(4, min(args.steps, 20))
    e0.record()
    for _ in range(e_steps):
        pipe.run(host, host_out)  # every step: H2D of its inputs, fw + bw kernels, D2H of its results
    pipe.flush()                  # (consecutive steps overlap on two device buffer sets; all of them end before e1)
    e1.record()
    sync_all()
    e2e_ms = replicas.max_over_ranks(e0.elapsed_time(e1), dev) / e_steps
    e2e_val = replicas.sum_over_ranks(ff + fb, dev) / (e2e_ms * 1e-3) / 1e12
    e2e_check = float((host_out["h"].float() - multi_out[0][0][0].float().cpu()).abs().max())  # same inputs as set 0

    del pipe
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    calls = None
    if world == 1 and not args.no_model_calls:
        calls = model_calls_block(pkg, dev, hbm_peak, flush)
    proxy = None
    if world > 1:
        proxy = ddp_proxy_block(pkg, dist, dev, world, flush)
    del flush
    mtrain = None
    if not args.no_model_train:
        mtrain = model_train_block(pkg, dist, dev, rank, world)
    minfer = model_infer_block(pkg, dev) if (world == 1 and not args.no_model_train) else None

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "TFLOP/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": WORKLOAD, "per_gpu": True, "kernel_impl": args.kernel_impl,
                       "l2": f"{N_SETS} rotating input sets, >126 MB touched between reuses (no explicit flush)",
                       "launch": f"CUDA graph replay, {N_SETS} steps (fw + bw kernels each, one per input set) per graph",
                       "frac_of_bf16_peak": value / world / tf_peak},
            "clocks": clocks, "gpu_launches": launches,
            "e2e": {"value": e2e_val, "unit": "TFLOP/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e_steps, "ms_per_step": e2e_ms, "api": "HostFwBw.run (pinned host in/out; per step H2D -> fw + bw kernels -> D2H on three streams as one CUDA graph; consecutive steps overlap on two device buffer sets)",
                    "max_abs_diff_vs_device_path": e2e_check},
            "roofline": roof,
            "dropin": dropin,
        }
        line["e2e"]["numa"] = numa
        line["e2e"]["note"] = ("PCIe-bound: %.0f MB in + %.0f MB out per step; every rank's pinned buffers sit on its GPU's NUMA node "
                               "when the platform reports one" % (h2d / 1e6, d2h / 1e6))
        if calls is not None:
            line["model_calls"] = calls
        if proxy is not None:
            line["ddp_proxy"] = proxy
        if mtrain is not None:
            line["model_train"] = mtrain
        if minfer is not None:
            line["model_infer"] = minfer
        if not args.no_cpu_baseline and world == 1:  # rank 0 at N = 1 only (at N > 1 the other ranks would spin in a barrier)
            line["cpu_baseline"] = cpu_baseline()
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
