#!/usr/bin/env python
"""Benchmark of the bridge hot path (BASELINE.json metric: bridge fwd+bwd samples/s; caption decode
tokens/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One "step" = one forward + backward of the bridge over one synthetic batch of config C2
(B=8 per GPU, L=128 text tokens, Nv=257 vision tokens, vision 1024 -> language 2304, 2 blocks,
heads 8/18, train mode with dropout 0.1 as `FullModel` builds it, full_model.py:38,72), upstream
gradient of loss = mean(y^2) (SURVEY.md 8d), bf16 weight copies refreshed every step as after an
optimizer update. Prints ONE JSON line (rank 0). See DESIGN.md "Measurement" for every field.

--dump-outputs DIR writes what the last timed step of the CUDA-graph replay (of the eager launches under
--no-graph) handed its caller, the loss and every parameter's gradient, as DIR/<name>.npy. Inputs, weights
and dropout seeds are fixed, so two builds run with the same arguments can be compared array for array.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# config C2 (BASELINE.json configs[1])
B_PER_GPU, L_TEXT, N_VIS, D_VIS, D_LANG, N_BLOCKS, H_CROSS, H_SELF = 8, 128, 257, 1024, 2304, 2, 8, 18
DROPOUT = 0.1
WORKLOAD = "C2"
# config C4 (decode): batch 32, 64 new tokens
DEC_B, DEC_STEPS = 32, 64


def gemm_flops_per_step(B: int, L: int, Nv: int) -> float:
    """Algorithmic FLOPs of the dense contractions (the tcgen05 GEMM kernel) in one fwd+bwd step:
    text-side linears forward + dgrad + wgrad, vision K/V projections forward + wgrad (SURVEY.md 8d)."""
    T, Tv, D, Dv, F = B * L, B * Nv, D_LANG, D_VIS, 4 * D_LANG
    text = N_BLOCKS * (2.0 * T * D * D * 6 + 4.0 * T * D * F)
    kv = N_BLOCKS * 4.0 * Tv * Dv * D
    return 3.0 * text + 2.0 * kv


def total_flops_per_step(B: int, L: int, Nv: int) -> float:
    T, D = B * L, D_LANG
    attn_fwd = N_BLOCKS * (4.0 * B * L * Nv * D + 4.0 * B * L * L * D)
    return gemm_flops_per_step(B, L, Nv) + 3.0 * attn_fwd


def decode_bytes_per_step(B: int, s: int, Nv: int, position_rows: bool = False) -> float:
    """Algorithmic HBM bytes of the decode cross-attention at prefix length s (bf16 cache):
    K and V of every block read once, Q read and O written (SURVEY.md 8d). With position rows
    block 0's launch has one query position (the new token) instead of s."""
    D = D_LANG
    lens = [1 if (position_rows and i == 0) else s for i in range(N_BLOCKS)]
    return sum(B * 2.0 * Nv * D * 2 + 2.0 * B * lq * D * 2 for lq in lens)


DUMP_ELEMS = 1 << 18   # per array: at most 52 x 1 MB of float32 in all


def step_outputs(loss, named_params) -> dict:
    """What one bridge step hands its caller, as float32 host arrays for --dump-outputs: the loss and the
    gradient of every parameter. A gradient of more than DUMP_ELEMS elements is sampled at DUMP_ELEMS flat
    positions drawn from a seed derived from the parameter's name, so every run samples the same positions."""
    import numpy as np
    import torch

    out = {"loss": loss.detach().float().reshape(1).cpu().numpy()}
    for name, p in named_params:
        g = p.grad.detach().reshape(-1)
        if g.numel() > DUMP_ELEMS:
            rng = np.random.default_rng(zlib.crc32(name.encode()))
            idx = np.sort(rng.choice(g.numel(), DUMP_ELEMS, replace=False))
            g = g[torch.from_numpy(idx).to(g.device)]
        out["grad." + name] = g.float().cpu().numpy()
    return out


def load_peaks() -> dict:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"bf16_burst": d.get("bf16_tflops", 1590.0), "bf16_sustained": d.get("bf16_tflops_sustained", 1400.0),
                "hbm": d.get("hbm_gbs", 6650.0), "source": "measured (MEASURED_PEAKS.json)"}
    return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms while a region runs."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None
        self.t0 = self.t1 = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu=timestamp,{self.FIELDS}",
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:  # noqa: BLE001
            self.proc = None

    def mark(self, begin: bool):
        if begin:
            self.t0 = time.time()
        else:
            self.t1 = time.time()

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        try:
            with open(self.path) as f:
                for line in f:
                    parts = [x.strip() for x in line.split(",")]
                    if len(parts) < 8:
                        continue
                    try:
                        sm.append(float(parts[1]))
                        mx.append(float(parts[2]))
                        power.append(float(parts[3]))
                    except ValueError:
                        continue
                    for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                         parts[4:8]):
                        if val.lower() == "active":
                            reasons.add(name)
            os.unlink(self.path)
        except Exception:  # noqa: BLE001
            pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # "under load": samples whose power draw is in the upper half of the observed range
        lo, hi = min(power), max(power)
        loaded = [s for s, p in zip(sm, power) if p >= lo + 0.5 * (hi - lo)] or sm
        return {"sm_mhz": statistics.median(loaded), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": hi}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference bridge on the host cores
# ------------------------------------------------------------------------------------------------
def _cpu_oracle():
    """The CPU restatement of the reference module: test infrastructure, imported by the CPU legs only."""
    from oracle import bridge_oracle as O

    return O


def cpu_decode_tokens_per_s(new_tokens: int = 16):
    """CPU baseline of caption decode (SURVEY.md 8d): the reference's loop shape -- batch 1, every step
    re-runs the bridge on the whole prefix INCLUDING the K/V projections of the unchanged image
    (full_model.py:241-256) -- bridge only, fp32, `new_tokens` steps from a 1-token prefix."""
    import torch

    O = _cpu_oracle()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = O.init_state_dict(0)
    g = torch.Generator().manual_seed(4321)
    vision = torch.randn(1, N_VIS, D_VIS, generator=g)
    text = torch.randn(1, new_tokens, D_LANG, generator=g)
    with torch.no_grad():
        O.bridge_forward(sd, vision, text[:, :1], num_blocks=N_BLOCKS, heads_cross=H_CROSS, heads_self=H_SELF)   # warm-up
        t0 = time.perf_counter()
        for s in range(1, new_tokens + 1):
            O.bridge_forward(sd, vision, text[:, :s], num_blocks=N_BLOCKS, heads_cross=H_CROSS, heads_self=H_SELF)
        dt = time.perf_counter() - t0
    return {"value": new_tokens / dt, "unit": "tokens/s", "cores": cores, "kind": "port",
            "sample": f"oracle port, batch 1, {new_tokens} new tokens, prefix and K/V projections recomputed every step "
                      f"(the reference's loop), fp32, bridge only; batch-1 latency-shaped: tokens/s of {DEC_B} images "
                      f"decoded one after the other is the same figure"}


def _cpu_reference_module():
    """The UNMODIFIED reference bridge_module.py, when oracle/make_ref.py has copied the reference package to
    oracle/_ref/ (git-ignored, travels to the GPU box); None otherwise."""
    try:
        from oracle import make_ref
        return make_ref.load_reference_bridge_module()
    except Exception:  # noqa: BLE001
        return None


def cpu_bridge_samples_per_s(steps: int, warmup: int, budget_s: float):
    """Times the reference's own CPU implementation of the path at config C2's shape on the host cores: the
    unmodified reference `BridgeLite` (oracle/_ref, train mode, dropout 0.1, fp32 -- `kind` "reference") when the
    copy is present, else the oracle port (eval mode: the port has no dropout -- `kind` "port").
    If a full batch-8 step would blow the time budget, a smaller batch is used as the sample and
    samples/s is computed from it (samples are independent in the bridge)."""
    import torch

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    g = torch.Generator().manual_seed(1234)
    ref = _cpu_reference_module()
    if ref is not None:
        torch.manual_seed(0)
        m = ref.BridgeLite(vision_dim=D_VIS, language_dim=D_LANG, num_blocks=N_BLOCKS, num_heads_cross=H_CROSS,
                           num_heads_self=H_SELF, dropout=DROPOUT).train()
        params = list(m.parameters())
        kind = "reference"
        what = (f"UNMODIFIED reference BridgeLite (oracle/_ref/vlm_bridge/model_architecture/bridge_module.py) fwd+bwd, "
                f"fp32, train mode dropout {DROPOUT}")

        def step(v, t):
            for p in params:
                p.grad = None
            m(v, t).square().mean().backward()
    else:
        O = _cpu_oracle()
        sd = O.init_state_dict(0)
        kind = "port"
        what = "oracle port of BridgeLite fwd+bwd (fp32, EVAL mode: the port has no dropout)"

        def step(v, t):
            O.bridge_loss_and_grads(sd, v, t, num_blocks=N_BLOCKS, heads_cross=H_CROSS, heads_self=H_SELF)

    def make(b):
        return torch.randn(b, N_VIS, D_VIS, generator=g), torch.randn(b, L_TEXT, D_LANG, generator=g)

    b = B_PER_GPU
    v, t = make(b)
    t0 = time.perf_counter()
    step(v, t)  # first call also pays allocator warm-up
    first = time.perf_counter() - t0
    total = steps + warmup
    if first * total > budget_s and b > 1:
        b = max(1, int(b * budget_s / (first * total)))
        v, t = make(b)
    for _ in range(max(0, warmup - 1)):
        step(v, t)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step(v, t)
        times.append(time.perf_counter() - t0)
    per_step = sum(times) / len(times)
    sample = (f"{what}, batch {b} x L{L_TEXT} x Nv{N_VIS}, "
              f"{steps} timed steps after {warmup} warm-up, torch CPU {torch.__version__}, {cores} threads")
    return b / per_step, per_step * 1e3, cores, sample, kind


def run_reference_arm(args) -> int:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    value, ms, cores, sample, kind = cpu_bridge_samples_per_s(args.steps, args.warmup, budget_s=200.0)
    line = {
        "impl": "reference", "metric": "bridge fwd+bwd samples/sec", "value": value, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


def workload_config(n_gpus: int) -> dict:
    return {
        "workload": (f"{WORKLOAD} bridge fwd+bwd: batch {B_PER_GPU}/GPU, text L={L_TEXT} x {D_LANG}, vision Nv={N_VIS} x {D_VIS}, "
                     f"{N_BLOCKS} blocks, heads {H_CROSS}/{H_SELF}, train mode dropout {DROPOUT}, loss=mean(y^2); "
                     "frozen DINOv2/Gemma are outside the hot path and not run"),
        "global_batch": B_PER_GPU * n_gpus,
        "parallelism": f"dp{n_gpus}" if n_gpus > 1 else "single",
        "l2": "working set (0.95 GB fp32+bf16 weights, 0.63 GB grads, >= 0.25 GB activations) exceeds the 126 MB L2; no flush needed",
        "weights": "random init (reference Xavier scheme, seed 0); bf16 copies re-cast every step",
        **({"gradients": "N > 1: bridge gradients averaged over ranks every step inside the backward (bf16 buckets over "
                         "NVLink / NVSwitch); the step's result is the averaged gradient in the form the fused optimizer "
                         "(BridgeAdamW) consumes: bf16 arena for the 2-D weights, fp32 for biases / LayerNorm "
                         "(--dp-fp32-grads adds the fp32 .grad materialisation pass); dp.parity_rel_err checks it against "
                         "the all-gathered mean of the per-rank gradients"} if n_gpus > 1 else {}),
    }


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def run_b200_arm(args) -> int:
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import datetime
        # a collective that a rank never joins aborts after 2 minutes instead of hanging the box
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=120))

    from vlm_bridge_b200 import BridgeLite, VisionKVCache, _lib
    from vlm_bridge_b200.parallel import broadcast_parameters, enable_data_parallel

    torch.manual_seed(0)
    model = BridgeLite(vision_dim=D_VIS, language_dim=D_LANG, num_blocks=N_BLOCKS, num_heads_cross=H_CROSS,
                       num_heads_self=H_SELF, dropout=DROPOUT).to(dev).train()
    params = list(model.parameters())
    g = torch.Generator().manual_seed(1234 + rank)
    vision_h = torch.randn(B_PER_GPU, N_VIS, D_VIS, generator=g).pin_memory()
    text_h = torch.randn(B_PER_GPU, L_TEXT, D_LANG, generator=g).pin_memory()
    vision_d, text_d = vision_h.to(dev), text_h.to(dev)
    torch.manual_seed(100 + rank)  # dropout seeds differ per rank
    if world > 1:
        with torch.no_grad():
            model(vision_d, text_d)  # flattens parameters
        broadcast_parameters(model)
        enable_data_parallel(model, grad_dtype=torch.float32 if args.grad_dtype == "f32" else torch.bfloat16,
                             backend=args.dp_backend, nvls_blocks=args.nvls_blocks, nvls_threads=args.nvls_threads,
                             bucket_bytes=args.bucket_mb << 20, exclusive_sms=args.nvls_exclusive,
                             fp32_multicast=args.nvls_fp32_multicast, nvls_unroll=args.nvls_unroll,
                             materialize_fp32=args.dp_fp32_grads)
        model._bucket_hook.diag_skip_convert = args.diag_dp_skip_convert
        model._bucket_hook.diag_skip_exchange = args.diag_dp_skip_exchange

    def step(v, t):
        model._w16_key = None            # weights count as updated by the optimizer since last step
        for p in params:
            p.grad = None
        y = model(v, t)
        loss = y.float().square().mean()
        loss.backward()
        return loss

    # The timed loops replay one captured CUDA graph of exactly this step (GraphedBridgeStep: forward,
    # loss, backward, weight re-cast, gradient exchange) unless --no-graph; the eager `step` remains for
    # the per-kernel event pass. Same kernels, same work; only the host-side enqueue cost differs.
    graphed, graph_error = None, None
    if not args.no_graph:
        from vlm_bridge_b200 import GraphedBridgeStep
        try:
            graphed = GraphedBridgeStep(model, lambda y: y.float().square().mean(), vision_d, text_d)
        except Exception as e:  # noqa: BLE001
            graph_error = repr(e)[:200]
            graphed = None
            torch.cuda.synchronize()

    def run_step(v, t):
        if graphed is None:
            return step(v, t)
        return graphed.replay() if v is vision_d else graphed(v, t)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    # --dump-outputs takes the last timed step of the launch mode the arguments fix: the graph replay, or the eager
    # launches under --no-graph (or when capture failed). Not the faster mode of the run: the two modes draw different
    # dropout seeds, and which one is faster can change from build to build.
    dump_mode = "eager launches" if graphed is None else "cuda graph replay (GraphedBridgeStep)"
    outputs = {}

    def timed_loop(fn, mode):
        for _ in range(max(3, args.warmup)):
            fn()
        sync_all()
        l0 = _lib.launch_count()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            loss = fn()
        host_ms = (time.perf_counter() - t0) * 1e3 / args.steps   # time to ENQUEUE a step (no sync inside)
        b.record()
        sync_all()
        if args.dump_outputs and mode == dump_mode:   # before the next loop overwrites them
            model.materialize_grads()      # N > 1: the averaged weight gradients out of the bf16 arena
            outputs[mode] = step_outputs(loss, model.named_parameters())
        ms = a.elapsed_time(b)
        if world > 1:                                              # a mode is as fast as its slowest rank
            tt_ = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(tt_, op=dist.ReduceOp.MAX)
            ms = float(tt_[0])
        return ms, host_ms, _lib.launch_count() - l0

    # ---- timed region: device-resident inputs. Both ways of launching the same step are timed (eager
    # launches with programmatic dependent launch, and one CUDA-graph replay per step); the faster is the
    # headline, both are reported ------------------------------------------------------------------
    sampler.mark(True)
    modes = {}
    if graphed is not None:
        mode = "cuda graph replay (GraphedBridgeStep)"
        ms_g, host_g, _ = timed_loop(lambda: graphed.replay(), mode)
        modes[mode] = (ms_g, host_g, graphed.kernels_per_replay * args.steps)
    if graphed is None or not args.graph_only:
        modes["eager launches"] = timed_loop(lambda: step(vision_d, text_d), "eager launches")
    sampler.mark(False)
    best_mode = min(modes, key=lambda k: modes[k][0])
    ms_total, host_ms_step, launches = modes[best_mode]
    if args.dump_outputs and rank == 0:
        import numpy as np

        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in outputs[dump_mode].items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    if best_mode == "eager launches":
        graphed_for_e2e, graphed = graphed, None                 # e2e and the dp leg follow the headline mode
    # ---- end-to-end: host buffers in, loss out, through the public nn.Module API ---------------
    # Every step's inputs travel from pinned host memory inside the timed region and every step's loss is
    # read back to the host. As a training loop with a pinned-memory loader does, the copy of step k+1's
    # inputs is issued on a copy stream while step k computes (two device buffers, events both ways).
    copy_stream = torch.cuda.Stream(device=dev)
    bufs = [(torch.empty_like(vision_d), torch.empty_like(text_d)) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]       # H2D of buffer i finished
    consumed = [torch.cuda.Event() for _ in range(2)]    # the step that read buffer i finished

    def prefetch(i):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[i])
            bufs[i][0].copy_(vision_h, non_blocking=True)
            bufs[i][1].copy_(text_h, non_blocking=True)
            ready[i].record(copy_stream)

    # Every step's loss is copied to pinned host memory right behind the step and read by the host one
    # step later (while the next step runs), as a training loop that logs its loss does to keep the GPU
    # fed: the host never waits on the step it has just launched.
    loss_host = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_done = [torch.cuda.Event() for _ in range(2)]

    def e2e_loop(n):
        cur = torch.cuda.current_stream()
        for c in consumed:
            c.record(cur)
        prefetch(0)
        out = 0.0
        for k in range(n):
            i = k & 1
            if k + 1 < n:
                prefetch(i ^ 1)
            cur.wait_event(ready[i])
            if graphed is not None:          # the graph's static input buffers <- device buffer, replay
                loss = graphed(bufs[i][0], bufs[i][1])
            else:
                loss = step(bufs[i][0], bufs[i][1])
            consumed[i].record(cur)
            loss_host[i].copy_(loss.detach().reshape(1), non_blocking=True)   # D2H of the step's result, every step
            loss_done[i].record(cur)
            if k > 0:
                loss_done[i ^ 1].synchronize()
                out += float(loss_host[i ^ 1])
        loss_done[(n - 1) & 1].synchronize()
        out += float(loss_host[(n - 1) & 1])
        return out

    def time_e2e():
        e2e_loop(3)
        sync_all()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        e2e_loop(args.steps)
        b.record()
        sync_all()
        ms = a.elapsed_time(b)
        if world > 1:
            tt_ = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(tt_, op=dist.ReduceOp.MAX)
            ms = float(tt_[0])
        return ms

    # with a host sync every step the enqueue cost of eager launches is exposed, so the graph replay can be
    # the faster way to run the SAME step end to end even when it is not for the device-resident loop
    e2e_modes = {}
    headline_graphed = graphed
    if best_mode == "eager launches":
        e2e_modes["eager launches"] = time_e2e()
        if graphed_for_e2e is not None:
            graphed = graphed_for_e2e
            e2e_modes["cuda graph replay (GraphedBridgeStep)"] = time_e2e()
            graphed = headline_graphed
    else:
        e2e_modes[best_mode] = time_e2e()
    e2e_mode = min(e2e_modes, key=lambda k: e2e_modes[k])

    ms_e2e_total = e2e_modes[e2e_mode]
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        tt = torch.tensor([ms_total, ms_e2e_total], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_total, ms_e2e_total = float(tt[0]), float(tt[1])
    ms_step = ms_total / args.steps
    ms_e2e = ms_e2e_total / args.steps
    value = B_PER_GPU * world / (ms_step * 1e-3)
    e2e_value = B_PER_GPU * world / (ms_e2e * 1e-3)

    line = {
        "metric": "bridge fwd+bwd samples/sec", "value": value, "unit": "samples/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": workload_config(world),
        "e2e": {"value": e2e_value, "unit": "samples/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": vision_h.numel() * 4 + text_h.numel() * 4, "d2h_bytes_per_step": 4,
                "launch_mode": e2e_mode, "ms_per_step_by_launch_mode": {k: v / args.steps for k, v in e2e_modes.items()},
                "how": "pinned host inputs copied H2D every step on a copy stream (double-buffered, overlapping the previous "
                       "step's compute); every step's loss copied D2H to pinned memory behind the step and read by the host "
                       "one step later (the last one after the loop, inside the timed region)"},
        "gpu_launches": int(launches),
        "host_enqueue_ms_per_step": host_ms_step,
        "launch_mode": best_mode + (f" (graph capture failed: {graph_error})" if graph_error else ""),
        "ms_per_step_by_launch_mode": {k: v[0] / args.steps for k, v in modes.items()},
        "pdl_mask": int(os.environ.get("B200B_PDL", "7")),
        "clocks": clocks,
    }

    if world > 1:
        # the same steps with the gradient exchange switched off: what the all-reduce costs per step
        from vlm_bridge_b200.parallel import disable_data_parallel
        reducer = model._bucket_hook
        disable_data_parallel(model)
        sync_all()
        e4, e5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        graphed_dp, graphed = graphed, None
        if graphed_dp is not None:
            try:
                graphed = GraphedBridgeStep(model, lambda y: y.float().square().mean(), vision_d, text_d)
            except Exception:  # noqa: BLE001
                graphed = None
        for _ in range(3):
            run_step(vision_d, text_d)
        sync_all()
        e4.record()
        t_host0 = time.perf_counter()
        for _ in range(args.steps):
            run_step(vision_d, text_d)
        host_ms_nodp = (time.perf_counter() - t_host0) * 1e3 / args.steps
        e5.record()
        sync_all()
        t_local = torch.tensor([e4.elapsed_time(e5)], device=dev, dtype=torch.float64)
        dist.all_reduce(t_local, op=dist.ReduceOp.MAX)
        model._bucket_hook = reducer
        graphed = graphed_dp
        trace = None
        if reducer.backend == "nvls":
            reducer.trace = []
            step(vision_d, text_d)
            bwd_end = torch.cuda.Event(enable_timing=True)
            bwd_end.record()
            torch.cuda.synchronize()
            trace = {"buckets": reducer.trace_report(), "backward_end_ms": round(reducer._t0.elapsed_time(bwd_end), 3)}
            reducer.trace = None
            sync_all()
        # ---- parity of the exchanged gradients at this N (untimed): eval mode (dropout off, so that the same
        # masks are not needed twice); want = mean over ranks of the no-exchange gradients (all-gathered through
        # NCCL in fp32); got = what every rank's .grad holds after a step with the exchange on, launched
        # eagerly and as a replay of a freshly captured graph
        def flat_grads():
            model.materialize_grads()          # no-op unless the exchange left the weight gradients in the bf16 arena
            return torch.cat([p.grad.detach().reshape(-1).float() for p in params])

        model.eval()
        model._bucket_hook = None
        step(vision_d, text_d)
        want = flat_grads().clone()
        dist.all_reduce(want, op=dist.ReduceOp.SUM)
        want /= world
        model._bucket_hook = reducer
        parity = {}
        step(vision_d, text_d)
        torch.cuda.synchronize()
        parity["eager"] = float((flat_grads() - want).norm() / want.norm())
        try:
            from vlm_bridge_b200 import GraphedBridgeStep
            gp = GraphedBridgeStep(model, lambda y: y.float().square().mean(), vision_d, text_d)
            gp.replay()
            gp.replay()
            torch.cuda.synchronize()
            parity["graph_replay"] = float((flat_grads() - want).norm() / want.norm())
            del gp
        except Exception as e:  # noqa: BLE001
            parity["graph_replay"] = repr(e)[:200]
        for p_ in params:
            p_.grad = None
        model.train()
        pt = torch.tensor([v if isinstance(v, float) else float("nan") for v in (parity["eager"], parity["graph_replay"])],
                          device=dev, dtype=torch.float64)
        dist.all_reduce(pt, op=dist.ReduceOp.MAX)                  # worst rank
        tol = 1.5e-2 if reducer.wgrad_bf16 else 1e-5
        parity_line = {"eager": float(pt[0]), "graph_replay": float(pt[1]), "tolerance": tol,
                       "ok": bool(float(pt[0]) <= tol and float(pt[1]) <= tol),
                       "what": "max over ranks of |grad_exchanged - mean_r grad_r| / |mean_r grad_r| (Frobenius, all 158 M "
                               "gradient elements), C2 shapes, eval mode; bf16 buckets round the weight gradients to bf16"}
        sync_all()
        line["dp"] = {"parity_rel_err": parity_line, "trace": trace, "allreduce": reducer.describe(), "bytes_per_step": reducer.bytes_per_step,
                      "ms_per_step_without_allreduce": float(t_local[0]) / args.steps,
                      "host_enqueue_ms_per_step_without_allreduce": host_ms_nodp,
                      "exposed_allreduce_ms": ms_step - float(t_local[0]) / args.steps}

    # ---- per-kernel timing pass (CUDA events on the launching stream, outside the timed region);
    # every rank runs the steps (they contain the gradient all-reduce), rank 0 records ----
    prof_steps = min(args.steps, 10)
    sync_all()
    if rank == 0:
        _lib.profile_begin(torch.cuda.current_stream().cuda_stream)
    for _ in range(prof_steps):
        step(vision_d, text_d)
    entries = _lib.profile_end() if rank == 0 else []
    sync_all()
    if rank == 0:
        peaks = load_peaks()
        # per kernel: total time within each profiled step, then the MEDIAN over the steps (an event pair
        # occasionally absorbs a host hiccup of milliseconds; a mean would carry it into the roofline)
        n_step = len(entries) // prof_steps
        per_step: list[dict[str, float]] = []
        counts: dict[str, int] = {}
        for s_i in range(prof_steps):
            acc: dict[str, float] = {}
            for name, ms in entries[s_i * n_step:(s_i + 1) * n_step]:
                acc[name] = acc.get(name, 0.0) + ms
                if s_i == 0:
                    counts[name] = counts.get(name, 0) + 1
            per_step.append(acc)
        kernel_ms = {k: statistics.median(d.get(k, 0.0) for d in per_step) for k in per_step[0]}
        gemm_names = [k for k in kernel_ms if k.startswith("gemm_tcgen05")]
        gemm_ms = sum(kernel_ms[k] for k in gemm_names)
        gemm_launches = sum(counts[k] for k in gemm_names)
        if os.environ.get("B200B_BENCH_DUMP"):
            with open(os.environ["B200B_BENCH_DUMP"], "w") as f:
                json.dump(entries[-n_step:], f)
        all_ms = sum(kernel_ms.values())
        gflops = gemm_flops_per_step(B_PER_GPU, L_TEXT, N_VIS)
        achieved = gflops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "r02_ncu_step_full.json")
        if os.path.exists(tp) and WORKLOAD == "C2":
            with open(tp) as f:
                traffic = json.load(f)["summary"]["dram_bytes_per_launch_avg"]
            traffic_src = ("profiles/r02_ncu_step_full.json: dram__bytes_read.sum + dram__bytes_write.sum of the 38 GEMM "
                           "launches of one step (ncu --set full capture of this round), average per launch")
        line["roofline"] = {
            "bound": "tensor", "kernel": "+".join(sorted(gemm_names)), "achieved": achieved, "peak": peaks["bf16_burst"],
            "unit": "TFLOP/s", "frac": achieved / peaks["bf16_burst"],
            "frac_of_sustained_peak": achieved / peaks["bf16_sustained"], "peak_sustained": peaks["bf16_sustained"],
            "peak_source": peaks["source"] + ", burst figure: the kernels are event-timed in a ~20 ms pass at full SM clock "
                           "(the sustained figure was taken under a power cap at 1357 MHz)", "traffic": traffic,
            "traffic_unit": "bytes per launch (HBM; the roofline itself is the tensor pipe)", "traffic_source": traffic_src,
            "launches_per_step": gemm_launches,
            "avg_launch_ms": gemm_ms / max(1, gemm_launches),
            "algorithmic_gflop_per_step": gflops / 1e9, "kernel_share_of_step": gemm_ms / all_ms if all_ms > 0 else None,
            "step_tflops_all_kernels": total_flops_per_step(B_PER_GPU, L_TEXT, N_VIS) / (ms_step * 1e-3) / 1e12,
            "kernel_ms_per_step": {k: v for k, v in sorted(kernel_ms.items())},
            "timing": "CUDA events recorded by the library after every launch on the launching stream, eager pass of "
                      f"{prof_steps} steps outside the timed region, median over steps",
        }
        # ---- decode (config C4): cached vision K/V, bridge-only loop. Decode shards images over the GPUs with no
        # communication ("replicas only"), so the leg belongs to the N = 1 line; at N > 1 it runs only with --decode
        # (the other ranks would sit in a collective while rank 0 works through it) --------------------------------
        if not args.no_decode and (world == 1 or args.decode):
            try:
                line["decode"] = bench_decode(model, dev, peaks, _lib)
            except Exception as e:  # noqa: BLE001
                line["decode"] = {"error": repr(e)[:300]}
        model.train()
        # ---- whole training step with the fused optimizer (SURVEY.md 8f rank 1), N=1 only ---------
        if world == 1 and not args.no_train_step:
            try:
                line["train_step"] = bench_train_step(model, step, vision_d, text_d, args.steps)
            except Exception as e:  # noqa: BLE001
                line["train_step"] = {"error": repr(e)[:300]}
        # ---- the same step through PyTorch's stock kernels on the same GPU (comparison), N=1 only ------
        if world == 1 and not args.no_train_step:
            try:
                line["torch_library"] = bench_torch_library(model, vision_d, text_d, args.steps)
            except Exception as e:  # noqa: BLE001
                line["torch_library"] = {"error": repr(e)[:300]}
        # ---- fused cross-entropy over the LM logits (SURVEY.md 8f rank 3), N=1 only ------------------
        if world == 1 and not args.no_train_step:
            try:
                line["fused_ce"] = bench_fused_ce(dev, peaks)
            except Exception as e:  # noqa: BLE001
                line["fused_ce"] = {"error": repr(e)[:300]}
        # ---- the bridge inside the unmodified reference training loop (SURVEY.md 8d C2(i)), N=1 only ----
        if world == 1 and not args.no_inloop:
            try:
                line["inloop"] = bench_inloop(args.steps)
            except Exception as e:  # noqa: BLE001
                line["inloop"] = {"error": repr(e)[:300]}
        # ---- CPU baseline beside it (N=1 only) ---------------------------------------------------
        if world == 1 and not args.no_cpu_baseline:
            v, ms, cores, sample, kind = cpu_bridge_samples_per_s(steps=3, warmup=1, budget_s=25.0)
            line["cpu_baseline"] = {"value": v, "unit": "samples/s", "cores": cores, "kind": kind, "sample": sample,
                                    "ms_per_step": ms}
            if isinstance(line.get("decode"), dict) and "error" not in line["decode"]:
                try:
                    line["decode"]["cpu_baseline"] = cpu_decode_tokens_per_s()
                except Exception as e:  # noqa: BLE001
                    line["decode"]["cpu_baseline"] = {"error": repr(e)[:200]}
        emit(line)
    if world > 1:
        # The last collective every rank takes part in is the barrier of sync_all() above; rank 0's remaining legs are
        # local. No final barrier / destroy_process_group(): a default N = 2 run of this file was seen to hang in that
        # tail after its JSON line had been written (profiles/r02 notes), so every rank leaves as soon as it is done --
        # the line went out through os.write, nothing buffered is lost.
        sys.stderr.flush()
        os._exit(0)
    return 0


def bench_train_step(model, step, vision_d, text_d, steps: int) -> dict:
    """fwd + bwd + BridgeAdamW.step (global-norm clip 0.3 + AdamW, config/training-default.yaml values), eager
    launches. The optimizer writes the bf16 operand copy of the weights, so the forward's re-cast pass is
    skipped -- unlike the headline step above, which re-casts every step to stand in for an optimizer."""
    import torch

    from vlm_bridge_b200 import BridgeAdamW

    opt = BridgeAdamW(model, lr=1e-5, weight_decay=0.01, max_grad_norm=0.3)
    params = list(model.parameters())

    def train_step():
        for p in params:
            p.grad = None
        loss = model(vision_d, text_d).float().square().mean()
        loss.backward()
        opt.step()
        return loss

    for _ in range(5):
        train_step()
    torch.cuda.synchronize()
    # one event per step, median over the steps: a single allocator / GC hiccup of ~100 ms was seen inside
    # this loop when it follows the other legs, and a mean would smear it over every step
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    evs[0].record()
    for i in range(steps):
        train_step()
        evs[i + 1].record()
    torch.cuda.synchronize()
    per = sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(steps))
    ms = per[len(per) // 2]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        opt.step()
    e1.record()
    torch.cuda.synchronize()
    ms_opt = e0.elapsed_time(e1) / steps
    return {"metric": "bridge training step samples/sec (fwd + bwd + fused clip/AdamW)", "value": B_PER_GPU / (ms * 1e-3),
            "unit": "samples/s", "ms_per_step": ms, "ms_per_step_mean": sum(per) / len(per), "ms_per_step_max": per[-1],
            "timing": "median of per-step CUDA-event intervals", "optimizer_ms": ms_opt,
            "optimizer_hbm_GBs": (158160384 * 32 + model._layout.n_weights * 2) / (ms_opt * 1e-3) / 1e9,
            "launch_mode": "eager", "grad_norm_last": float(opt.last_grad_norm),
            "steps_that_gathered_grads": opt.gather_steps}


def torch_library_forward(sd, vision, text, num_blocks: int, heads_cross: int, heads_self: int, p: float, training: bool):
    """The bridge arithmetic spelled with PyTorch's stock operators (F.linear -> cuBLASLt, F.layer_norm,
    F.scaled_dot_product_attention, F.gelu, F.dropout) over a BridgeLite `state_dict`: what the same GPU does
    for this workload WITHOUT this repository's kernels. Used only as a timed comparison (`torch_library` in the
    bench line) and checked against the oracle on the CPU (tests/test_bench_contract.py)."""
    import torch.nn.functional as F

    def lin(x, name):
        return F.linear(x, sd[name + ".weight"], sd[name + ".bias"])

    def norm(x, name):
        return F.layer_norm(x, x.shape[-1:], sd[name + ".weight"], sd[name + ".bias"], 1e-5)

    def mha(q, k, v, h):
        def split(t):
            return t.view(t.shape[0], t.shape[1], h, t.shape[2] // h).transpose(1, 2)
        o = F.scaled_dot_product_attention(split(q), split(k), split(v), dropout_p=p if training else 0.0)
        return o.transpose(1, 2).reshape(q.shape)

    x = text
    for i in range(num_blocks):
        b = f"bridge_blocks.{i}."
        xn = norm(x, b + "ln_cross")
        c = b + "cross_attention."
        x = x + lin(mha(lin(xn, c + "w_q"), lin(vision, c + "w_k"), lin(vision, c + "w_v"), heads_cross), c + "w_o")
        xn = norm(x, b + "ln_self")
        a = b + "self_attention."
        x = x + lin(mha(lin(xn, a + "w_q"), lin(xn, a + "w_k"), lin(xn, a + "w_v"), heads_self), a + "w_o")
        xn = norm(x, b + "ln_ffn")
        hidden = F.dropout(F.gelu(lin(xn, b + "ffn.0")), p, training)
        x = x + F.dropout(lin(hidden, b + "ffn.3"), p, training)
    return x


def bench_torch_library(model, vision_d, text_d, steps: int) -> dict:
    """The same fwd+bwd step on the same GPU through PyTorch's own kernels under torch.autocast(bfloat16) -- how
    the reference module itself would run on this B200. Timed twice: eager launches (what the reference's loop
    does; may be host-bound) and as a replay of one captured CUDA graph (device time only: the like-for-like
    figure against this repository's graph replay). A comparison line, not a target."""
    import torch

    sd = {k: v.detach().clone().requires_grad_() for k, v in model.state_dict().items()}
    leaves = list(sd.values())

    def step(set_none=True):
        if set_none:
            for t in leaves:
                t.grad = None
        with torch.autocast("cuda", dtype=torch.bfloat16):
            y = torch_library_forward(sd, vision_d, text_d, N_BLOCKS, H_CROSS, H_SELF, DROPOUT, True)
        loss = y.float().square().mean()
        loss.backward()
        return loss

    def timed(fn, n):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    n = max(5, min(20, steps))
    ms = timed(step, n)
    ms_graph, graph_err = None, None
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        for t in leaves:
            t.grad = None
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            step(set_none=False)          # grads are allocated from the graph's pool and overwritten per replay
        ms_graph = timed(gr.replay, n)
        del gr
    except Exception as e:  # noqa: BLE001
        graph_err = repr(e)[:200]
        torch.cuda.synchronize()
    best = min(ms, ms_graph) if ms_graph is not None else ms
    return {"metric": "bridge fwd+bwd samples/sec through PyTorch's stock kernels on the same GPU", "value": B_PER_GPU / (best * 1e-3),
            "unit": "samples/s", "ms_per_step": best, "steps": n,
            "ms_per_step_by_launch_mode": {"eager": ms, "cuda graph replay": ms_graph, "graph_error": graph_err},
            "how": f"torch {torch.__version__}, torch.autocast(bfloat16): F.linear (cuBLASLt), F.layer_norm, "
                   "F.scaled_dot_product_attention, F.gelu, F.dropout; same weights, inputs, dropout p, loss"}


def bench_inloop(steps: int) -> dict:
    """BASELINE.json configs[1] / SURVEY.md 8d C2(i): the full training step of the UNMODIFIED reference
    (`run_training_epoch`, core_training_loop.py:16-134: FullModel.forward under autocast(bf16), CE over the 256000-token
    vocabulary, GradScaler, the per-parameter gradient-norm loop, clip_grad_norm_, AdamW) at batch 8, caption length
    128, 224 px, random-init frozen DINOv2-large + Gemma-2-2B (full depth), timed with this repository's BridgeLite
    swapped in and with the reference's own bridge. Wall clock per step (the loop synchronises with the host 50+
    times per step). Needs oracle/_ref (oracle/make_ref.py) and transformers; reports why if it cannot run."""
    import torch

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import inloop_harness as H

    ok, why = H.available()
    if not ok:
        return {"unavailable": why}
    from vlm_bridge_b200 import BridgeLite

    with H.quiet():
        model = H.build_full_model(BridgeLite, bridge_dropout=DROPOUT)
    from vlm_bridge.training_strategy.core_training_loop import run_training_epoch

    ours = model.bridge_module
    ref_bridge = H.reference_bridge_cls()(vision_dim=D_VIS, language_dim=D_LANG, num_heads_cross=H_CROSS, dropout=DROPOUT).to("cuda")
    ref_bridge.load_state_dict(ours.state_dict(), strict=True)
    n = max(3, min(8, steps))
    batches = H.make_batches(n, B_PER_GPU, L_TEXT)
    out = {}
    legs = (("b200_bridge", ours), ("reference_bridge_torch_eager", ref_bridge))
    opts = {}
    for name, bridge in legs:                              # warm-up: 2 steps each (cuBLAS heuristics, allocator)
        model.bridge_module = bridge
        ctx = H.training_context(model, batches[:2])
        with H.quiet():
            run_training_epoch(ctx, 0)
        opts[name] = ctx.optimizer
    # the frozen models dominate the step (~95 %) and run-to-run variation is a few ms: the legs alternate and the
    # fastest epoch of each is reported
    for rep in range(3):
        for name, bridge in legs:
            model.bridge_module = bridge
            ctx = H.training_context(model, batches, optimizer=opts[name])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            with H.quiet():
                loss = run_training_epoch(ctx, 1 + rep)
            torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) * 1e3 / n
            if name not in out or ms < out[name]["ms_per_step"]:
                out[name] = {"ms_per_step": ms, "avg_loss": loss}
    # the bridge's own share: fwd + bwd of the swapped-in module at the same shapes, device time
    g = torch.Generator().manual_seed(1)
    v = torch.randn(B_PER_GPU, N_VIS, D_VIS, generator=g).cuda()
    t = torch.randn(B_PER_GPU, L_TEXT, D_LANG, generator=g).cuda().requires_grad_()
    share = {}
    for name, bridge in (("b200_bridge", ours), ("reference_bridge_torch_eager", ref_bridge)):
        bridge.train()

        def one():
            with torch.autocast("cuda", dtype=torch.bfloat16):
                y = bridge(v, t)
            y.float().square().mean().backward()

        for _ in range(3):
            one()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            one()
        e1.record()
        torch.cuda.synchronize()
        share[name] = e0.elapsed_time(e1) / n
    res = {"metric": "full training step of the unmodified reference loop, ms per step (wall clock)",
           "config": f"B{B_PER_GPU} L{L_TEXT} 224 px, random-init frozen DINOv2-large (24 layers) + Gemma-2-2B (26 layers), "
                     f"bf16 autocast + GradScaler + clip 0.3 + torch AdamW, best of 3 alternating epochs of {n} steps after 2 warm-up steps",
           "whole_step_ms": {k: v_["ms_per_step"] for k, v_ in out.items()},
           "avg_loss": {k: v_["avg_loss"] for k, v_ in out.items()},
           "bridge_fwd_bwd_ms_same_shapes_eager": share,
           "samples_per_s": {k: B_PER_GPU / (v_["ms_per_step"] * 1e-3) for k, v_ in out.items()}}
    del model, ours, ref_bridge
    torch.cuda.empty_cache()
    return res


def bench_fused_ce(dev, peaks) -> dict:
    """Loss of the C2 training step: [B*L, V] = [1024, 256000] fp32 logits (what autocast hands
    cross_entropy), labels shifted in-kernel; fwd + bwd timed with CUDA events, HBM roofline on the
    algorithmic bytes (logits read twice, gradient written once). torch's own loss timed beside it."""
    import torch
    import torch.nn.functional as F

    from vlm_bridge_b200 import FusedCrossEntropyLoss

    rows, L, V = B_PER_GPU * L_TEXT, L_TEXT, 256000
    g = torch.Generator().manual_seed(99)
    logits = torch.randn(rows, V, generator=g).to(dev).requires_grad_()
    ids = torch.randint(3, V, (B_PER_GPU, L), generator=g).to(dev)
    labels = ids.clone()
    labels[:, :-1] = ids[:, 1:]
    labels[:, -1] = -100
    loss_fn = FusedCrossEntropyLoss()

    def ours():
        logits.grad = None
        loss_fn.forward_shifted(logits, ids).backward()

    def theirs():
        logits.grad = None
        F.cross_entropy(logits, labels.view(-1), ignore_index=-100).backward()

    out = {}
    for name, fn in (("fused", ours), ("torch", theirs)):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out[name] = e0.elapsed_time(e1) / reps
    nbytes = 3.0 * rows * V * 4
    achieved = nbytes / (out["fused"] * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "r01_ncu_ce_summary.json")
    if os.path.exists(tp):
        with open(tp) as f:
            traffic = json.load(f)["summary"]["dram_bytes_fwd_plus_bwd"]
        traffic_src = "profiles/r01_ncu_ce_summary.json: dram__bytes_read.sum + dram__bytes_write.sum, forward + backward launches"
    return {"metric": "cross-entropy fwd+bwd over [1024, 256000] fp32 logits", "ms": out["fused"], "torch_ms": out["torch"],
            "roofline": {"bound": "hbm", "kernel": "ce_fwd_kernel + ce_bwd_kernel", "achieved": achieved,
                         "peak": peaks["hbm"], "unit": "GB/s", "frac": achieved / peaks["hbm"],
                         "algorithmic_bytes": nbytes, "traffic": traffic, "traffic_source": traffic_src},
            "note": "inputs (2.1 GB with the gradient) exceed the 126 MB L2; includes the autograd node overhead"}


def decode_gemm_flops(B: int, steps: int, Nv: int, position_rows: bool = True) -> float:
    """Algorithmic FLOPs of the dense contractions of one caption batch (steps new tokens, prefix s = 1..steps):
    the per-image K/V projection once, block 0's cross-attention projections once per position (position rows) or
    once per position per step, everything else of both blocks over the whole prefix every step."""
    D, Dv, F = D_LANG, D_VIS, 4 * D_LANG
    per_row_cross = 2.0 * D * D * 2                       # w_q, w_o
    per_row_rest = 2.0 * D * D * 4 + 4.0 * D * F          # self q,k,v,o + ffn
    rows_all = B * steps * (steps + 1) / 2.0
    rows_new = B * steps
    total = N_BLOCKS * 2.0 * (B * Nv) * Dv * D * 2        # K and V of every block
    total += per_row_cross * ((rows_new if position_rows else rows_all) + (N_BLOCKS - 1) * rows_all)
    total += per_row_rest * N_BLOCKS * rows_all
    return total


def bench_decode(model, dev, peaks, _lib) -> dict:
    """Config C4: batched greedy caption decode, batch 32, 64 new tokens, through `greedy_decode` itself (embed ->
    bridge over the prefix -> read-out -> argmax -> append, ids read back). The frozen language model is outside
    the hot path; a fixed embedding table and a fixed linear read-out (vocabulary 8192) stand in for it. Every
    caption batch pays the per-image K/V projection + packing (`VisionKVCache` built, or refilled in place when
    the step graphs are reused)."""
    import torch

    from vlm_bridge_b200 import DecodeStepGraphs, VisionKVCache, greedy_decode

    model.eval()
    V = 8192
    g = torch.Generator().manual_seed(4321)
    vision_h = torch.randn(DEC_B, N_VIS, D_VIS, generator=g).pin_memory()
    vision = vision_h.to(dev)
    embed = torch.randn(V, D_LANG, generator=g).to(dev)
    head = (torch.randn(V, D_LANG, generator=g) / 48.0).to(dev)
    ids_h = torch.empty((DEC_B, DEC_STEPS + 1), dtype=torch.long).pin_memory()
    kw = dict(bos_token_id=2, eos_token_id=1, max_new_tokens=DEC_STEPS)

    def e_fn(t):
        return embed[t]

    def l_fn(h):
        return h[:, -1, :] @ head.t()

    def timed(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    # eager launches; a new cache per caption batch
    ms_eager = timed(lambda: greedy_decode(model, vision, e_fn, l_fn, **kw))
    # one CUDA graph of the bridge per prefix length, captured ONCE; every caption batch refills the cache in place
    cache = VisionKVCache(model, vision)
    graphs = DecodeStepGraphs(model, cache)
    ms_graph, graph_err = None, None
    try:
        ms_graph = timed(lambda: greedy_decode(model, vision, e_fn, l_fn, kv_cache=cache, step_graphs=graphs,
                                               refill_cache=True, **kw))
    except Exception as e:  # noqa: BLE001
        graph_err = repr(e)[:200]
    use_graphs = ms_graph is not None and ms_graph < ms_eager
    ms = ms_graph if use_graphs else ms_eager

    # end to end: image features from pinned host memory in, token ids to the host out, every caption batch
    def e2e_once():
        v = vision_h.to(dev, non_blocking=True)
        if use_graphs:
            ids, _ = greedy_decode(model, v, e_fn, l_fn, kv_cache=cache, step_graphs=graphs, refill_cache=True, **kw)
        else:
            ids, _ = greedy_decode(model, v, e_fn, l_fn, **kw)
        ids_h.copy_(ids, non_blocking=True)
        torch.cuda.synchronize()          # the caller needs the ids
    ms_e2e = timed(e2e_once)
    # variants (eager): no position rows; no cache at all (what the reference does: re-project K/V every step)
    ms_kv_only = timed(lambda: greedy_decode(model, vision, e_fn, l_fn, cache_positions=False, **kw))
    ms_uncached = timed(lambda: greedy_decode(model, vision, e_fn, l_fn, use_cache=False, **kw), reps=1)
    # kernel-level: this library's launches of one caption batch (eager pass, events after every launch)
    _lib.profile_begin(torch.cuda.current_stream().cuda_stream)
    greedy_decode(model, vision, e_fn, l_fn, **kw)
    entries = _lib.profile_end()
    per_kernel: dict[str, float] = {}
    for name, ms_ in entries:
        per_kernel[name] = per_kernel.get(name, 0.0) + ms_
    cross_ms = sum(v for k, v in per_kernel.items() if k in ("attn_decode_packed", "attn_decode_tc"))
    gemm_ms = sum(v for k, v in per_kernel.items() if k.startswith("gemm_tcgen05"))
    bytes_total = sum(decode_bytes_per_step(DEC_B, s, N_VIS, position_rows=True) for s in range(1, DEC_STEPS + 1))
    achieved_eager = bytes_total / (cross_ms * 1e-3) / 1e9 if cross_ms > 0 else 0.0
    # The same 128 cross-attention launches of one caption batch (block 0: 1 new position per step; block 1: the
    # whole prefix; same kernels, same cache, same shapes) back to back in ONE CUDA graph, timed with CUDA events:
    # the kernels' own duration, without the gaps an event pair sees between eager launches of a host-bound loop.
    from vlm_bridge_b200 import ops
    from vlm_bridge_b200.bridge import TC_DECODE_MIN_LEN
    Hc, dk = H_CROSS, D_LANG // H_CROSS
    qbuf = torch.randn(DEC_B * DEC_STEPS, D_LANG, generator=torch.Generator().manual_seed(5)).bfloat16().to(dev)
    obuf = torch.empty_like(qbuf)

    def cross_launches():
        for s_ in range(1, DEC_STEPS + 1):
            for blk, lq in ((0, 1), (1, s_)):
                kw_ = dict(block_index=blk, num_blocks=N_BLOCKS, batch=DEC_B, heads=Hc, len_q=lq, len_k=N_VIS, head_dim=dk,
                           out=obuf[:DEC_B * lq], want_lse=False)
                if lq >= TC_DECODE_MIN_LEN:
                    ops.attention_decode_tc(qbuf[:DEC_B * lq], cache.kv_tc, **kw_)
                else:
                    ops.attention_decode_packed(qbuf[:DEC_B * lq], cache.kv_packed, **kw_)

    cross_launches()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        cross_launches()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    cg = torch.cuda.CUDAGraph()
    with torch.cuda.graph(cg):
        cross_launches()
    cg.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        cg.replay()
    e1.record()
    torch.cuda.synchronize()
    cross_ms_graph = e0.elapsed_time(e1) / 5
    del cg
    achieved = bytes_total / (cross_ms_graph * 1e-3) / 1e9
    gflop = decode_gemm_flops(DEC_B, DEC_STEPS, N_VIS)
    gemm_tf = gflop / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "r01_ncu_decode_packed_summary.json")
    if os.path.exists(tp):
        with open(tp) as f:
            traffic = json.load(f)["summary"]["dram_bytes_per_launch_len_q_1"]
        traffic_src = ("profiles/r01_ncu_decode_packed_summary.json: dram__bytes_read.sum + dram__bytes_write.sum of one "
                       "1-position launch (ncu --set full); algorithmic bytes of that launch: 76.1 MB")
    tok = DEC_B * DEC_STEPS
    return {
        "metric": "caption decode tokens/sec (greedy_decode: embed + bridge + read-out + argmax; cached vision K/V)",
        "value": tok / (ms * 1e-3), "unit": "tokens/s", "ms_per_caption_batch": ms,
        "launch_mode": "graph replay per prefix length, cache refilled in place per caption batch" if use_graphs else "eager launches",
        "ms_per_caption_batch_by_launch_mode": {"eager (new VisionKVCache per caption batch)": ms_eager,
                                                "graph replay (graphs captured once; K/V projection + packing refilled "
                                                "in place per caption batch)": ms_graph, "graph_error": graph_err},
        "e2e": {"value": tok / (ms_e2e * 1e-3), "unit": "tokens/s", "ms_per_caption_batch": ms_e2e,
                "h2d_bytes_per_step": vision_h.numel() * 4, "d2h_bytes_per_step": ids_h.numel() * 8,
                "how": "per caption batch: image features H2D from pinned memory, greedy_decode, token ids D2H, host sync"},
        "uncached_tokens_per_s": tok / (ms_uncached * 1e-3),
        "kv_cache_only_tokens_per_s": tok / (ms_kv_only * 1e-3),
        "config": (f"C4: batch {DEC_B}, {DEC_STEPS} new tokens, Nv={N_VIS}; vision K/V cached per image, block 0's "
                   "cross-attention rows cached per text position, everything from block 0's non-causal "
                   f"self-attention on recomputed over the prefix every step; stand-in LM: embedding table + linear "
                   f"read-out, vocabulary {V}"),
        "roofline": {"bound": "hbm", "kernel": "attn_decode_kernel<288, packed> for <= 32 positions (all 64 block-0 launches: 1 position each), attn_decode_tc_kernel<288> above (the 128 cross-attention launches)", "achieved": achieved,
                     "peak": peaks["hbm"], "unit": "GB/s", "frac": achieved / peaks["hbm"], "traffic": traffic,
                     "traffic_source": traffic_src, "algorithmic_bytes_total": bytes_total, "kernel_ms_total": cross_ms_graph,
                     "avg_launch_ms": cross_ms_graph / (2 * DEC_STEPS), "launches": 2 * DEC_STEPS,
                     "timing": "the 128 launches of one caption batch back to back in one CUDA graph, CUDA events around 5 "
                               "replays (the cache, 156 MB, exceeds the 126 MB L2)",
                     "achieved_event_timed_in_eager_loop": achieved_eager, "kernel_ms_total_event_timed_in_eager_loop": cross_ms,
                     "note": "the eager figure includes the idle gaps between launches of the host-bound Python loop"},
        "gemm_roofline": {"bound": "tensor", "kernel": "gemm_tcgen05 (prefix recompute: M = 32 * s rows)",
                          "achieved": gemm_tf, "peak": peaks["bf16_burst"], "unit": "TFLOP/s",
                          "frac": gemm_tf / peaks["bf16_burst"], "algorithmic_tflop_per_caption_batch": gflop / 1e12,
                          "kernel_ms_total": gemm_ms},
        "kernel_ms_per_caption_batch": {k: round(v, 4) for k, v in sorted(per_kernel.items())},
        "kv_cache_bytes": cache.nbytes,
    }


_JSON_FD = None


def own_stdout() -> None:
    """The contract is ONE JSON line on stdout. Libraries write there too (NCCL prints its version banner to
    fd 1 on some boxes), so fd 1 is pointed at stderr for the rest of the run and the JSON line goes to a
    private duplicate of the original stdout."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _JSON_FD is None:
        os.write(1, data)
    else:
        os.write(_JSON_FD, data)


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-decode", action="store_true")
    ap.add_argument("--decode", action="store_true", help="run the decode leg at N > 1 as well (default: N = 1 only)")
    ap.add_argument("--no-train-step", action="store_true")
    ap.add_argument("--no-inloop", action="store_true", help="skip the leg that runs the unmodified reference training loop")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches only (no CUDA-graph replay)")
    ap.add_argument("--graph-only", action="store_true", help="time the CUDA-graph replay only")
    ap.add_argument("--dp-backend", default="auto", choices=["auto", "nvls", "nccl"],
                    help="transport of the gradient exchange: own NVLS multimem kernel, or NCCL")
    ap.add_argument("--nvls-blocks", type=int, default=16)
    ap.add_argument("--nvls-threads", type=int, default=1024)
    ap.add_argument("--nvls-exclusive", action="store_true", help="reserve --nvls-blocks SMs for the exchange")
    ap.add_argument("--nvls-unroll", type=int, default=8, choices=[4, 8, 16], help="16-byte units in flight per thread")
    ap.add_argument("--dp-fp32-grads", action="store_true",
                    help="N > 1: materialise fp32 .grad tensors every step (one more bf16 -> fp32 pass over 158 M elements). "
                         "Default: the averaged weight gradients stay in the bf16 arena, which is what BridgeAdamW consumes "
                         "(module.materialize_grads() produces fp32 .grad on demand)")
    ap.add_argument("--nvls-fp32-multicast", action="store_true", help="broadcast fp32 into .grad (no conversion pass)")
    ap.add_argument("--diag-dp-skip-convert", action="store_true",
                    help="diagnostics: skip the bf16 -> fp32 pass of the exchange (gradients are then incomplete)")
    ap.add_argument("--diag-dp-skip-exchange", action="store_true",
                    help="diagnostics: launch no collective (what writing the gradients into the symmetric arenas costs by itself)")
    ap.add_argument("--bucket-mb", type=int, default=32)
    ap.add_argument("--grad-dtype", default="bf16", choices=["bf16", "f32"],
                    help="dtype of the data-parallel weight-gradient exchange (N > 1)")
    ap.add_argument("--workload", default="c2", choices=["c2", "c5"],
                    help="c2 = BASELINE.json configs[1] (the headline, default); c5 = the 518 px stress config "
                         "(batch 16, 1370 vision tokens), bridge fwd+bwd only")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss and the parameter gradients of the last timed graph replay (eager step under "
                         "--no-graph) as DIR/<name>.npy (float32; "
                         f"gradients of more than {DUMP_ELEMS} elements sampled at fixed seeded positions)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.workload == "c5":
        global B_PER_GPU, N_VIS, WORKLOAD
        B_PER_GPU, N_VIS, WORKLOAD = 16, 1370, "C5"
        args.no_decode = args.no_train_step = args.no_cpu_baseline = args.no_inloop = True
    own_stdout()
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_b200_arm(args)


if __name__ == "__main__":
    sys.exit(main())
