"""Cost of top-k sampling and of several sampled captions per image: the fused sampler with top_k (csrc/sampling.cu)
against the PyTorch recipe on the same buffers, its top_k = 0 path against the top-p-only entry point, and a C4
caption batch sampled with num_return_sequences = 5 over the shared cache against the images repeated 5 times.

  python tests/gpu_checks/exp_topk_multi.py [--out PATH]   (needs a CUDA device; default PATH
                                                            profiles/r05_exp_topk_multi.jsonl)

Kernel cases: rows = 32 x V = 256 000 x {fp32, bf16} x top_k in {50, 1000, 32000} x top_p in {1.0, 0.9}, temperature
0.8. Each case rotates through enough logits buffers that they total more than 160 MB, above the 126 MB L2, so every
launch reads its logits from HBM. The sampler is timed as a CUDA-graph replay of 96 launches (one buffer each in turn);
the PyTorch recipe (guards, divide, topk + mask, then for top_p < 1 sort, softmax, cumsum, mask, scatter; softmax,
multinomial: the order of Hugging Face's warpers) is timed eagerly over the same buffers, alternating with the sampler,
five rounds each, medians reported.

top_k = 0 against the old entry: the same [32, 256 000] cases at top_p 1.0 / 0.9, b200b_sample_tokens_top_k(top_k = 0)
and b200b_sample_tokens each captured as a graph of 96 launches, replayed alternately for 9 rounds; medians, minima
and maxima of each are reported, so a difference can be read against the spread of the same code.

Caption batch: C4 (32 images, 64 new tokens, 257 vision tokens, real widths, bf16 bridge, graphs over a refilled
cache), stand-in language model with a 256 000-row read-out, do_sample (T 0.8, top_k 50, top_p 0.9): N = 5 over
VisionKVCache(beams=5) against the same decode over vision.repeat_interleave(5, 0), timed alternately, three rounds
each after a warm-up call that captures the graphs. Cross-attention K/V bytes per step are counted from the layout
each block's kernel reads (block 0 computes the new row of every sequence, the later blocks the whole prefix), at
prefix 16 and summed over the 64 steps.
"""
from __future__ import annotations

import ctypes as C
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
ROWS = 32
HBM_PEAK = 7.7e12
L2_BYTES = 126e6
GRAPH_LAUNCHES = 96
N_SEQ = 5


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[0] if q.stdout else
            f"nvidia-smi failed: {q.stderr.strip()[:200]}"}


def time_events(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def torch_recipe(x, temperature, top_k, top_p):
    x = x.float()
    bad = torch.isnan(x).any(dim=-1, keepdim=True)
    x = torch.where(bad, torch.zeros_like(x), x)
    x = torch.where(torch.isinf(x).any(dim=-1, keepdim=True), x.clamp(min=-100, max=100), x)
    z = x / temperature
    z = z.masked_fill(z < torch.topk(z, top_k, dim=-1).values[..., -1:], -math.inf)
    if top_p < 1.0:
        sz, order = torch.sort(z, descending=True, dim=-1)
        p = torch.softmax(sz, dim=-1)
        cum = torch.cumsum(p, dim=-1)
        sz = sz.masked_fill(cum - p >= top_p, -math.inf)
        z = torch.empty_like(z).scatter_(1, order, sz)
    return torch.multinomial(torch.softmax(z, dim=-1), 1)


def _buffers(dt, seed):
    esz = 4 if dt == torch.float32 else 2
    nbytes = ROWS * V * esz
    nbuf = max(2, math.ceil(160e6 / nbytes))
    g = torch.Generator(device="cuda").manual_seed(seed)
    return [(torch.randn(ROWS, V, device="cuda", generator=g) * 3.0).to(dt) for _ in range(nbuf)], nbytes


def _graph(launch):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            for i in range(GRAPH_LAUNCHES):
                launch(i)
    torch.cuda.current_stream().wait_stream(s)
    graph.replay()
    torch.cuda.synchronize()
    return graph


def kernel_case(dt, top_k, top_p, temperature=0.8):
    from vlm_bridge_b200 import ops

    bufs, nbytes = _buffers(dt, top_k)
    nbuf = len(bufs)
    seed = torch.tensor([11], dtype=torch.int64, device="cuda")
    out = torch.empty(ROWS, dtype=torch.int64, device="cuda")
    for bb in bufs[:2]:
        ops.sample_tokens(bb, temperature=temperature, top_k=top_k, top_p=top_p, seed=seed, step=0, out=out)
        torch_recipe(bb, temperature, top_k, top_p)
    torch.cuda.synchronize()
    graph = _graph(lambda i: ops.sample_tokens(bufs[i % nbuf], temperature=temperature, top_k=top_k, top_p=top_p,
                                               seed=seed, step=i, out=out))
    k_ms, t_ms = [], []
    n_torch = max(nbuf, 20)
    for _ in range(5):
        k_ms.append(time_events(graph.replay, 3) / GRAPH_LAUNCHES)
        it = iter(range(10 ** 9))
        t_ms.append(time_events(lambda: torch_recipe(bufs[next(it) % nbuf], temperature, top_k, top_p), n_torch))
    km, tm = sorted(k_ms)[2], sorted(t_ms)[2]
    return {"kind": "sampler_top_k", "status": "measured", "rows": ROWS, "vocab": V,
            "dtype": "fp32" if dt == torch.float32 else "bf16", "top_k": top_k, "top_p": top_p,
            "temperature": temperature, "buffers": nbuf, "buffer_mb_total": round(nbuf * nbytes / 1e6, 1),
            "l2_mb": L2_BYTES / 1e6, "reads_from": "HBM (rotating buffers larger than L2)", "bytes": nbytes,
            "kernel_us": round(km * 1e3, 2), "kernel_us_rounds": [round(v * 1e3, 2) for v in k_ms],
            "hbm_fraction_of_7.7TBs": round(nbytes / (km * 1e-3) / HBM_PEAK, 3),
            "torch_recipe_us": round(tm * 1e3, 2), "torch_recipe_us_rounds": [round(v * 1e3, 2) for v in t_ms],
            "speedup_vs_torch": round(tm / km, 2)}


def entry_case(dt, top_p, temperature=0.8, rounds=9):
    """b200b_sample_tokens_top_k(top_k = 0) against b200b_sample_tokens, graphs replayed alternately."""
    from vlm_bridge_b200 import _lib

    lib = _lib.lib()
    bufs, nbytes = _buffers(dt, 99)
    nbuf = len(bufs)
    seed = torch.tensor([11], dtype=torch.int64, device="cuda")
    outs = {w: torch.empty(ROWS, dtype=torch.int64, device="cuda") for w in ("old", "new")}
    dtc = 1 if dt == torch.bfloat16 else 0

    def launch(which, i):
        x = bufs[i % nbuf]
        stream = torch.cuda.current_stream().cuda_stream
        if which == "old":
            rc = lib.b200b_sample_tokens(x.data_ptr(), dtc, x.stride(0), ROWS, V, temperature, top_p, seed.data_ptr(),
                                         i, outs[which].data_ptr(), 1, stream)
        else:
            rc = lib.b200b_sample_tokens_top_k(x.data_ptr(), dtc, x.stride(0), ROWS, V, temperature, 0, top_p,
                                               seed.data_ptr(), i, outs[which].data_ptr(), 1, stream)
        _lib.check(rc, which)

    graphs = {w: _graph(lambda i, w=w: launch(w, i)) for w in ("old", "new")}
    same = bool(torch.equal(outs["old"], outs["new"]))
    ms = {w: [] for w in graphs}
    for _ in range(rounds):
        for w, g in graphs.items():
            ms[w].append(time_events(g.replay, 3) / GRAPH_LAUNCHES * 1e3)
    med = {w: sorted(v)[rounds // 2] for w, v in ms.items()}
    return {"kind": "top_k0_vs_old_entry", "status": "measured", "rows": ROWS, "vocab": V,
            "dtype": "fp32" if dt == torch.float32 else "bf16", "top_p": top_p, "temperature": temperature,
            "reads_from": "HBM (rotating buffers larger than L2)", "ids_equal": same,
            "old_entry_us": round(med["old"], 2), "old_entry_us_min_max": [round(min(ms["old"]), 2), round(max(ms["old"]), 2)],
            "new_entry_top_k0_us": round(med["new"], 2),
            "new_entry_top_k0_us_min_max": [round(min(ms["new"]), 2), round(max(ms["new"]), 2)],
            "old_entry_us_rounds": [round(v, 2) for v in ms["old"]],
            "new_entry_top_k0_us_rounds": [round(v, 2) for v in ms["new"]],
            "new_minus_old_us": round(med["new"] - med["old"], 2)}


def cross_kv_bytes(m, cache, L):
    """K/V bytes the cross-attention of one cached decode step at prefix L reads, per block from the layout that
    block's kernel reads (BridgeLite._kv_flag of its query rows per image): block 0 computes the new row of each
    sequence (beams rows per image), the later blocks the whole prefix (beams * L rows). Each layout holds every
    block, so one block reads 1 / num_blocks of it."""
    total = 0
    for i in range(m.num_blocks):
        rows = cache.beams * (1 if i == 0 else L)
        kv_t, _ = m._kv_flag(cache, rows, False)
        total += kv_t.numel() * kv_t.element_size() // m.num_blocks
    return total


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
    ef, lf = (lambda t: embed[t]), (lambda y: y[:, -1, :] @ head.t())
    rep = vision.repeat_interleave(N_SEQ, 0)
    shared = VisionKVCache(m, vision, max_positions=STEPS, beams=N_SEQ)
    repl = VisionKVCache(m, rep, max_positions=STEPS)
    gs, gr = DecodeStepGraphs(m, shared), DecodeStepGraphs(m, repl)
    gen = torch.Generator(device="cuda")
    kw = dict(bos_token_id=2, eos_token_id=1, max_new_tokens=STEPS, refill_cache=True, do_sample=True, temperature=0.8,
              top_k=50, top_p=0.9, generator=gen)

    def run(which):
        gen.manual_seed(5)
        if which == "shared":
            return greedy_decode(m, vision, ef, lf, num_return_sequences=N_SEQ, kv_cache=shared, step_graphs=gs, **kw)
        return greedy_decode(m, rep, ef, lf, kv_cache=repl, step_graphs=gr, **kw)

    a, b = run("shared"), run("replicated")
    torch.cuda.synchronize()
    ms = {"shared": [], "replicated": []}
    for _ in range(3):
        for w in ms:
            ms[w].append(time_events(lambda: run(w), 1))
    out = {"kind": "caption_batch_num_return_sequences", "status": "measured",
           "config": "C4: B 32, 64 new tokens, 257 vision tokens, bf16 bridge, graphs over a refilled cache",
           "lm": "stand-in: embedding table + fp32 linear read-out, V = 256000",
           "num_return_sequences": N_SEQ, "temperature": 0.8, "top_k": 50, "top_p": 0.9,
           "same_shape": tuple(a[0].shape) == tuple(b[0].shape),
           "rows_equal_to_replicated": int((a[0] == b[0]).all(dim=1).sum()), "rows": int(a[0].shape[0])}
    for w, cache in (("shared", shared), ("replicated", repl)):
        out[f"{w}_ms"] = round(sorted(ms[w])[1], 2)
        out[f"{w}_ms_rounds"] = [round(v, 2) for v in ms[w]]
        out[f"{w}_cross_kv_bytes_per_step_at_prefix16"] = cross_kv_bytes(m, cache, 16)
        out[f"{w}_cross_kv_bytes_64_steps"] = sum(cross_kv_bytes(m, cache, L) for L in range(1, STEPS + 1))
    return out


def main():
    if not torch.cuda.is_available():
        raise SystemExit("exp_topk_multi.py needs a CUDA device")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    lines = [dict(kind="card", sms=sms, **card())]
    print(json.dumps(lines[-1]), flush=True)
    for dt in (torch.float32, torch.bfloat16):
        for top_p in (1.0, 0.9):
            lines.append(entry_case(dt, top_p))
            print(json.dumps(lines[-1]), flush=True)
            torch.cuda.empty_cache()
    for dt in (torch.float32, torch.bfloat16):
        for top_k in (50, 1000, 32000):
            for top_p in (1.0, 0.9):
                lines.append(kernel_case(dt, top_k, top_p))
                print(json.dumps(lines[-1]), flush=True)
                torch.cuda.empty_cache()
    lines.append(caption_case())
    print(json.dumps(lines[-1]), flush=True)
    lines.append(dict(kind="card_after", **card()))
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else os.path.join(ROOT, "profiles",
                                                                                        "r05_exp_topk_multi.jsonl")
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
