"""Cost of beam search: the fused beam step (csrc/beam.cu) against the PyTorch recipe on the same buffers, the bridge
step over a shared per-image cache against a replicated one, and a C4 caption batch with K = 4 against greedy.

  python tests/gpu_checks/exp_beam.py [--out PATH]   (needs a CUDA device; default PATH profiles/r04_exp_beam.jsonl)

Beam step: rows = 32 images x 4 beams, V = 256 000, fp32 and bf16 logits. Each case rotates through enough logits
buffers that they total more than 160 MB, above the 126 MB L2, so every step reads its logits from HBM. The beam
step (two launches) is timed as a CUDA-graph replay of 96 steps (one buffer each in turn); the PyTorch recipe
(log_softmax in fp32, add the beam scores, view(B, K*V).topk(2K), parent / token split, gather of the first K
beams' ids and scores: less than the full rule, which also walks the EOS candidates) is timed eagerly over the same
buffers, alternating with the kernel, five rounds each, medians reported. Bytes = rows * V * e (e = 4 fp32, 2 bf16),
the least the step must read, over time, as a fraction of the 7.7 TB/s data-sheet HBM bandwidth.

Bridge step: 32 images x 4 beams, bf16, one decode step at prefix length 16 with the cached position rows (block 0
computes the new row only), replayed from a captured graph. Shared cache: VisionKVCache(beams=4) over the 32 images;
replicated: a cache of the images repeated 4 times. Cross-attention bytes per step = the K/V each block's
cross-attention reads, from the layout its kernel reads (block 0: one new row per beam; later blocks: the whole
prefix of every beam, so 64 query rows per image read the tcgen05 layout on the shared cache).

Caption batch: C4 (32 images, 64 new tokens, 257 vision tokens, real widths, bf16 bridge, graphs over a refilled
cache), stand-in language model with a 256 000-row read-out; greedy and beam search (K = 4, EOS 1, length penalty 1)
timed alternately, three rounds each after a warm-up call that captures the graphs.
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
B, K = 32, 4
HBM_PEAK = 7.7e12
L2_BYTES = 126e6
GRAPH_STEPS = 96


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


def torch_recipe(x, scores, ids, t):
    lp = torch.log_softmax(x.float(), dim=-1) + scores[:, None]
    top_s, top_i = lp.view(B, K * V).topk(2 * K, dim=-1)
    parent = top_i // V + torch.arange(B, device=x.device)[:, None] * K
    token = top_i % V
    nxt = ids.index_select(0, parent[:, :K].reshape(-1))
    nxt[:, t + 1] = token[:, :K].reshape(-1)
    return nxt, top_s[:, :K].reshape(-1)


def kernel_case(dt):
    from vlm_bridge_b200 import ops

    esz = 4 if dt == torch.float32 else 2
    rows = B * K
    nbytes = rows * V * esz
    nbuf = max(2, math.ceil(160e6 / nbytes))
    g = torch.Generator(device="cuda").manual_seed(esz)
    bufs = [(torch.randn(rows, V, device="cuda", generator=g) * 3.0).to(dt) for _ in range(nbuf)]
    t = 3
    ids = torch.randint(0, V, (rows, t + 2), device="cuda", generator=g)
    ids_next = torch.empty_like(ids)
    parents = torch.empty(rows, dtype=torch.int64, device="cuda")
    st = ops.BeamState(B, K, t + 2, "cuda")
    st.beam_scores.copy_(-torch.rand(rows, device="cuda", generator=g) * 5)
    scores = st.beam_scores.clone()

    def step(i):
        ops.beam_step(bufs[i % nbuf], ids, ids_next, parents, st, step=t, eos_token_id=1, length_penalty=1.0)

    for i in range(2):
        step(i)
        torch_recipe(bufs[i], scores, ids, t)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            for i in range(GRAPH_STEPS):
                step(i)
    torch.cuda.current_stream().wait_stream(s)
    graph.replay()
    torch.cuda.synchronize()
    k_ms, t_ms = [], []
    n_torch = max(nbuf, 20)
    for _ in range(5):
        k_ms.append(time_events(graph.replay, 3) / GRAPH_STEPS)
        it = iter(range(10 ** 9))
        t_ms.append(time_events(lambda: torch_recipe(bufs[next(it) % nbuf], scores, ids, t), n_torch))
    km, tm = sorted(k_ms)[2], sorted(t_ms)[2]
    return {"kind": "beam_step", "images": B, "beams": K, "rows": rows, "vocab": V,
            "dtype": "fp32" if esz == 4 else "bf16", "buffers": nbuf, "buffer_mb_total": round(nbuf * nbytes / 1e6, 1),
            "l2_mb": L2_BYTES / 1e6, "reads_from": "HBM (rotating buffers larger than L2)", "bytes": nbytes,
            "kernel_us": round(km * 1e3, 2), "kernel_us_rounds": [round(v * 1e3, 2) for v in k_ms],
            "hbm_fraction_of_7.7TBs": round(nbytes / (km * 1e-3) / HBM_PEAK, 3),
            "torch_recipe_us": round(tm * 1e3, 2), "torch_recipe_us_rounds": [round(v * 1e3, 2) for v in t_ms],
            "speedup_vs_torch": round(tm / km, 2)}


def _model():
    from oracle import bridge_oracle as O
    from vlm_bridge_b200 import BridgeLite

    m = BridgeLite(dropout=0.0)
    m.load_state_dict(O.init_state_dict(1), strict=True)
    return m.cuda().eval()


def cross_kv_bytes(m, cache, L):
    """K/V bytes the cross-attention of one cached decode step at prefix L reads, per block from the layout that
    block's kernel reads (BridgeLite._kv_flag of its query rows per image): block 0 computes the new row of each
    beam (beams rows per image), the later blocks the whole prefix (beams * L rows). Each layout holds every block,
    so one block reads 1 / num_blocks of it."""
    names = {id(cache.kv): "projection output", id(cache.kv_packed): "packed (mma.sync)"}
    if cache.kv_tc is not None:
        names[id(cache.kv_tc)] = "tcgen05 tiles"
    total, used = 0, []
    for i in range(m.num_blocks):
        rows = cache.beams * (1 if i == 0 else L)
        kv_t, _ = m._kv_flag(cache, rows, False)
        total += kv_t.numel() * kv_t.element_size() // m.num_blocks
        used.append(f"block {i}: {rows} query rows per image -> {names[id(kv_t)]}")
    return total, used


def bridge_step_case():
    from vlm_bridge_b200 import VisionKVCache
    from vlm_bridge_b200.decode import DecodeStepGraphs

    L = 16
    m = _model()
    g = torch.Generator(device="cuda").manual_seed(3)
    vision = torch.randn(B, 257, 1024, device="cuda", generator=g)
    text = torch.randn(B * K, L, 2304, device="cuda", generator=g)
    out = {"kind": "bridge_step", "images": B, "beams": K, "prefix_len": L, "precision": "bf16",
           "cached_positions": L - 1, "timing": "graph replay, median of 5 rounds of 20"}
    caches = {"shared": VisionKVCache(m, vision, beams=K), "replicated": VisionKVCache(m, vision.repeat_interleave(K, 0))}
    runs = {}
    with torch.no_grad():
        for name, cache in caches.items():
            m(None, text[:, :L - 1], kv_cache=cache, cached_positions=0)
            graphs = DecodeStepGraphs(m, cache)
            graphs(text, cached_positions=L - 1)
            runs[name] = graphs
            out[f"{name}_cross_kv_bytes_per_step"], out[f"{name}_cross_kv_layouts"] = cross_kv_bytes(m, cache, L)
        torch.cuda.synchronize()
        ms = {n: [] for n in runs}
        for _ in range(5):
            for name, graphs in runs.items():
                ms[name].append(time_events(lambda: graphs(text, cached_positions=L - 1), 20))
    for name in runs:
        out[f"{name}_step_ms"] = round(sorted(ms[name])[2], 4)
        out[f"{name}_step_ms_rounds"] = [round(v, 4) for v in ms[name]]
    return out


def caption_case():
    from vlm_bridge_b200 import VisionKVCache, beam_search_decode, greedy_decode
    from vlm_bridge_b200.decode import DecodeStepGraphs

    STEPS = 64
    g = torch.Generator(device="cuda").manual_seed(20)
    vision = torch.randn(B, 257, 1024, device="cuda", generator=g)
    embed = torch.randn(V, 2304, device="cuda", generator=g)
    head = torch.randn(V, 2304, device="cuda", generator=g) / 48.0
    m = _model()
    ef, lf = (lambda t: embed[t]), (lambda y: y[:, -1, :] @ head.t())
    gc = VisionKVCache(m, vision, max_positions=STEPS)
    gg = DecodeStepGraphs(m, gc)
    bc = VisionKVCache(m, vision, max_positions=STEPS, beams=K)
    bg = DecodeStepGraphs(m, bc)
    kw = dict(bos_token_id=2, eos_token_id=1, max_new_tokens=STEPS, refill_cache=True)

    def run(beam):
        if beam:
            return beam_search_decode(m, vision, ef, lf, num_beams=K, kv_cache=bc, step_graphs=bg, **kw)
        return greedy_decode(m, vision, ef, lf, kv_cache=gc, step_graphs=gg, **kw)

    run(False)
    run(True)
    torch.cuda.synchronize()
    gr, be = [], []
    for _ in range(3):
        gr.append(time_events(lambda: run(False), 1))
        be.append(time_events(lambda: run(True), 1))
    return {"kind": "caption_batch", "config": "C4: B 32, 64 new tokens, 257 vision tokens, bf16 bridge, graphs",
            "lm": "stand-in: embedding table + fp32 linear read-out, V = 256000",
            "greedy_ms": round(sorted(gr)[1], 2), "greedy_ms_rounds": [round(v, 2) for v in gr],
            "beam4_ms": round(sorted(be)[1], 2), "beam4_ms_rounds": [round(v, 2) for v in be]}


def main():
    if not torch.cuda.is_available():
        raise SystemExit("exp_beam.py needs a CUDA device")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    lines = [dict(kind="card", sms=sms, **card())]
    print(json.dumps(lines[-1]), flush=True)
    for dt in (torch.float32, torch.bfloat16):
        lines.append(kernel_case(dt))
        print(json.dumps(lines[-1]), flush=True)
        torch.cuda.empty_cache()
    lines.append(bridge_step_case())
    print(json.dumps(lines[-1]), flush=True)
    torch.cuda.empty_cache()
    lines.append(caption_case())
    print(json.dumps(lines[-1]), flush=True)
    lines.append(dict(kind="card_after", **card()))
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else os.path.join(ROOT, "profiles",
                                                                                        "r04_exp_beam.jsonl")
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
