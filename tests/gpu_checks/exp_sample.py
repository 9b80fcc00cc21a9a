"""Cost of temperature / top-p sampling over a 256 000-entry vocabulary: the fused sampler (csrc/sampling.cu)
against the stock PyTorch recipe on the same buffers, and one C4 caption batch sampled against greedy.

  python tests/gpu_checks/exp_sample.py [--out PATH]   (needs a CUDA device; default PATH profiles/r03_exp_sample.jsonl)

Kernel cases: rows in {1, 32, 64} x V = 256 000 x {fp32, bf16} x top_p in {1.0, 0.9}, temperature 0.8. Each case
rotates through enough logits buffers that they total more than 160 MB, above the 126 MB L2, so every launch reads
its logits from HBM. The sampler is timed as a CUDA-graph replay of 96 launches (one launch per buffer in turn;
a rows = 1 launch is shorter than its eager enqueue); the PyTorch recipe (guards, divide, sort, softmax, cumsum,
mask, scatter, softmax, multinomial; the filter is skipped at top_p = 1 as a caller would) is timed eagerly over
the same buffers, alternating with the sampler, five rounds each, medians reported. Bytes = rows * V * e (e = 4
fp32, 2 bf16) over time, as a fraction of the 7.7 TB/s data-sheet HBM bandwidth.

The cluster size each case runs with is the library's rule (include/b200_bridge.h), restated below: bf16 rows = 32
and rows = 64 fall on the two sides of its SM-coverage doubling.

Caption batch: C4 (32 images, 64 new tokens, 257 vision tokens, real widths, bf16 bridge, graphs over a refilled
cache) with a stand-in language model whose read-out has 256 000 rows; greedy and do_sample=True (T 0.8, top_p
0.9) timed alternately, three rounds each after a warm-up call that captures the graphs.
"""
from __future__ import annotations

import json
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

V = 256000
HBM_PEAK = 7.7e12
L2_BYTES = 126e6
GRAPH_LAUNCHES = 96


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else
            f"nvidia-smi failed: {q.stderr.strip()[:200]}"}


def cluster_size(rows, vocab, esz, sms):
    """b200b_sample_tokens' rule: fewest CTAs whose slices fit 176 KiB, doubled while rows * CTAs < SMs and each
    CTA keeps >= 4096 tokens (at most 8)."""
    def fits(c):
        return ((vocab + c - 1) // c + 7) // 8 * 8 * esz <= 176 * 1024
    c = 1
    while not fits(c):
        c *= 2
    while c < 8 and rows * c < sms and vocab >= 2 * c * 4096:
        c *= 2
    return c


def torch_recipe(x, temperature, top_p):
    x = x.float()
    bad = torch.isnan(x).any(dim=-1, keepdim=True)
    x = torch.where(bad, torch.zeros_like(x), x)
    x = torch.where(torch.isinf(x).any(dim=-1, keepdim=True), x.clamp(min=-100, max=100), x)
    z = x / temperature
    if top_p < 1.0:
        sz, order = torch.sort(z, descending=True, dim=-1)
        p = torch.softmax(sz, dim=-1)
        cum = torch.cumsum(p, dim=-1)
        sz = sz.masked_fill(cum - p >= top_p, -math.inf)
        z = torch.empty_like(z).scatter_(1, order, sz)
    return torch.multinomial(torch.softmax(z, dim=-1), 1)


def time_events(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def kernel_case(rows, dt, top_p, sms, temperature=0.8):
    from vlm_bridge_b200 import ops

    esz = 4 if dt == torch.float32 else 2
    nbytes = rows * V * esz
    nbuf = max(2, math.ceil(160e6 / nbytes))
    g = torch.Generator(device="cuda").manual_seed(rows)
    bufs = [(torch.randn(rows, V, device="cuda", generator=g) * 3.0).to(dt) for _ in range(nbuf)]
    seed = torch.tensor([11], dtype=torch.int64, device="cuda")
    out = torch.empty(rows, dtype=torch.int64, device="cuda")
    for bb in bufs[:2]:
        ops.sample_tokens(bb, temperature=temperature, top_p=top_p, seed=seed, step=0, out=out)
        torch_recipe(bb, temperature, top_p)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            for i in range(GRAPH_LAUNCHES):
                ops.sample_tokens(bufs[i % nbuf], temperature=temperature, top_p=top_p, seed=seed, step=i, out=out)
    torch.cuda.current_stream().wait_stream(s)
    graph.replay()
    torch.cuda.synchronize()
    k_ms, t_ms = [], []
    n_torch = max(nbuf, 20)
    for _ in range(5):
        k_ms.append(time_events(graph.replay, 3) / GRAPH_LAUNCHES)
        it = iter(range(10 ** 9))
        t_ms.append(time_events(lambda: torch_recipe(bufs[next(it) % nbuf], temperature, top_p), n_torch))
    km, tm = sorted(k_ms)[2], sorted(t_ms)[2]
    return {"kind": "kernel", "rows": rows, "vocab": V, "dtype": "fp32" if esz == 4 else "bf16", "top_p": top_p,
            "temperature": temperature, "cluster_ctas": cluster_size(rows, V, esz, sms),
            "buffers": nbuf, "buffer_mb_total": round(nbuf * nbytes / 1e6, 1), "l2_mb": L2_BYTES / 1e6,
            "reads_from": "HBM (rotating buffers larger than L2)",
            "bytes": nbytes, "kernel_us": round(km * 1e3, 2), "kernel_us_rounds": [round(v * 1e3, 2) for v in k_ms],
            "hbm_fraction_of_7.7TBs": round(nbytes / (km * 1e-3) / HBM_PEAK, 3),
            "torch_recipe_us": round(tm * 1e3, 2), "torch_recipe_us_rounds": [round(v * 1e3, 2) for v in t_ms],
            "speedup_vs_torch": round(tm / km, 2)}


def caption_case():
    from oracle import bridge_oracle as O
    from vlm_bridge_b200 import BridgeLite, VisionKVCache, greedy_decode
    from vlm_bridge_b200.decode import DecodeStepGraphs

    B, NV, STEPS = 32, 257, 64
    g = torch.Generator(device="cuda").manual_seed(20)
    vision = torch.randn(B, NV, 1024, device="cuda", generator=g)
    embed = torch.randn(V, 2304, device="cuda", generator=g)
    head = torch.randn(V, 2304, device="cuda", generator=g) / 48.0
    m = BridgeLite(dropout=0.0)
    m.load_state_dict(O.init_state_dict(1), strict=True)
    m = m.cuda().eval()
    cache = VisionKVCache(m, vision, max_positions=STEPS)
    graphs = DecodeStepGraphs(m, cache)
    gen = torch.Generator(device="cuda").manual_seed(5)
    kw = dict(bos_token_id=2, eos_token_id=1, max_new_tokens=STEPS, kv_cache=cache, step_graphs=graphs,
              refill_cache=True)

    def run(sample):
        if sample:
            return greedy_decode(m, vision, lambda t: embed[t], lambda y: y[:, -1, :] @ head.t(), do_sample=True,
                                 temperature=0.8, top_p=0.9, generator=gen, **kw)
        return greedy_decode(m, vision, lambda t: embed[t], lambda y: y[:, -1, :] @ head.t(), **kw)

    run(False)
    run(True)
    torch.cuda.synchronize()
    gr, sa = [], []
    for _ in range(3):
        gr.append(time_events(lambda: run(False), 1))
        sa.append(time_events(lambda: run(True), 1))
    return {"kind": "caption_batch", "config": "C4: B 32, 64 new tokens, 257 vision tokens, bf16 bridge, graphs",
            "lm": "stand-in: embedding table + fp32 linear read-out, V = 256000",
            "greedy_ms": round(sorted(gr)[1], 2), "greedy_ms_rounds": [round(v, 2) for v in gr],
            "do_sample_ms": round(sorted(sa)[1], 2), "do_sample_ms_rounds": [round(v, 2) for v in sa],
            "temperature": 0.8, "top_p": 0.9}


def main():
    if not torch.cuda.is_available():
        raise SystemExit("exp_sample.py needs a CUDA device")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    lines = [dict(kind="card", sms=sms, **card())]
    print(json.dumps(lines[-1]), flush=True)
    for rows in (1, 32, 64):
        for dt in (torch.float32, torch.bfloat16):
            for top_p in (1.0, 0.9):
                lines.append(kernel_case(rows, dt, top_p, sms))
                print(json.dumps(lines[-1]), flush=True)
                torch.cuda.empty_cache()
    lines.append(caption_case())
    print(json.dumps(lines[-1]), flush=True)
    lines.append(dict(kind="card_after", **card()))
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else os.path.join(ROOT, "profiles",
                                                                                        "r03_exp_sample.jsonl")
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
