"""Batched caption decode over a per-image cached vision K/V (SURVEY.md 8a row a12, 8f rank 2).

Mirrors `FullModel.generate_caption` (full_model.py:241-363); the greedy branch (`do_sample=False`):
start from BOS, every step embeds the whole prefix, runs the bridge over it (the bridge
self-attention is non-causal, so earlier positions change when a token is appended and the prefix
must be recomputed -- only the image's K/V are exactly cacheable), feeds the result to the language
model, takes `argmax` of the last position's logits (NaN logits -> zeros, Inf logits -> clamped to
+-100, as :270-283) and appends it. With `do_sample=True` the token is drawn instead (temperature, top-k,
top-p nucleus, one fused kernel per step: `ops.sample_tokens`, csrc/sampling.cu), as the sampling branch
(:264-350) does; `num_return_sequences` draws several captions per image over one shared cache of the image.

The reference loop is batch-1 and synchronises with the host up to three times per step
(`next_token.item()`, :317,355-366). Here B images decode together with no host synchronisation:
every row runs `max_new_tokens` steps and is cut at its first EOS afterwards, which is what B
independent reference runs produce (generation is deterministic and rows never interact).

`embed_fn` / `lm_fn` stand for the frozen language model, which is outside the hot path:
`embed_fn(ids [B, s]) -> [B, s, D]` (LanguageModel.get_embeddings, language_model.py:146-164) and
`lm_fn(hidden [B, s, D]) -> logits [B, s, V]` or `[B, V]` for the last position
(LanguageModel.forward_from_embeddings, :111-144).
"""
from __future__ import annotations

import math
import numbers
from typing import Callable, Optional

import torch

from . import ops
from .kv_cache import VisionKVCache

__all__ = ["greedy_decode", "beam_search_decode", "DecodeStepGraphs"]


class DecodeStepGraphs:
    """One captured CUDA graph of the bridge forward per (batch, prefix length), over a fixed
    `VisionKVCache`: a decode step is ~45 short kernels, so enqueueing them from Python takes longer
    than they run; a replay costs one launch. The graphs share a memory pool (they never run
    concurrently) and are valid while the cache is (`VisionKVCache.is_current()`); the bf16 weight
    copies are NOT re-cast inside these graphs (inference: the weights are frozen)."""

    def __init__(self, bridge, kv_cache: VisionKVCache):
        self.bridge, self.cache = bridge, kv_cache
        self._graphs: dict = {}
        self._pool = None

    def __call__(self, text_embeddings: torch.Tensor, cached_positions: Optional[int] = None) -> torch.Tensor:
        """bridge(vision, text_embeddings, kv_cache=cache, cached_positions=...) for text_embeddings
        [B, s, D]; the returned tensor is the graph's static output (overwritten by the next call with
        the same shape)."""
        if not self.cache.is_current():
            raise RuntimeError("the K/V cache is stale (bridge weights changed): rebuild it and the graphs")
        key = (int(text_embeddings.shape[0]), int(text_embeddings.shape[1]), cached_positions)
        if cached_positions is not None:
            # the host-side bookkeeping a replay skips (also validates the request)
            if self.cache.position_rows(key[1], cached_positions, text_embeddings.device, text_embeddings.shape[-1]) is None:
                key = key[:2] + (None,)
                cached_positions = None
        ent = self._graphs.get(key)
        if ent is None:
            b = self.bridge
            static_in = text_embeddings.detach().to(torch.float32).clone()
            with torch.no_grad():
                b(None, static_in, kv_cache=self.cache, cached_positions=cached_positions)   # lazy init outside the capture
                torch.cuda.synchronize()
                if self._pool is None:
                    self._pool = torch.cuda.graph_pool_handle()
                g = torch.cuda.CUDAGraph()
                recast, b._graph_recast = b._graph_recast, False
                try:
                    with torch.cuda.graph(g, pool=self._pool):
                        out = b(None, static_in, kv_cache=self.cache, cached_positions=cached_positions)
                finally:
                    b._graph_recast = recast
            ent = self._graphs[key] = (g, static_in, out)
        g, static_in, out = ent
        static_in.copy_(text_embeddings, non_blocking=True)
        g.replay()
        return out


def _decode_setup(bridge, vision_features, max_new_tokens, kv_cache, use_cache, step_graphs, use_graphs, precision,
                  refill_cache, beams: int = 1):
    """The argument, cache and graph setup of the decode drivers: (kv_cache, step_graphs) to use."""
    if precision not in ("bf16", "fp32"):
        raise ValueError("precision must be 'bf16' or 'fp32'")
    if precision == "fp32" and not use_cache:
        raise RuntimeError("precision='fp32' reads an fp32 VisionKVCache: use_cache must stay True")
    if kv_cache is not None and use_cache and getattr(kv_cache, "beams", 1) != beams:
        raise ValueError(f"kv_cache was built for beams={kv_cache.beams}, this decode runs {beams}")
    if use_cache and kv_cache is None:
        kv_cache = VisionKVCache(bridge, vision_features, precision=precision, max_positions=max(64, max_new_tokens),
                                 beams=beams)
    elif use_cache:
        if kv_cache.precision != precision:
            raise RuntimeError(f"kv_cache holds {kv_cache.precision} K/V but precision={precision!r} was asked for")
        if refill_cache:
            kv_cache.refill(vision_features)
    if (use_graphs or step_graphs is not None) and use_cache:
        if step_graphs is None or step_graphs.cache is not kv_cache:
            step_graphs = DecodeStepGraphs(bridge, kv_cache)
    else:
        step_graphs = None
    return kv_cache, step_graphs


@torch.no_grad()
def greedy_decode(bridge, vision_features: torch.Tensor, embed_fn: Callable[[torch.Tensor], torch.Tensor],
                  lm_fn: Callable[[torch.Tensor], torch.Tensor], *, bos_token_id: int,
                  eos_token_id: Optional[int] = None, max_new_tokens: int = 50,
                  kv_cache: Optional[VisionKVCache] = None, use_cache: bool = True,
                  step_graphs: Optional[DecodeStepGraphs] = None, use_graphs: bool = False,
                  cache_positions: bool = True, precision: str = "bf16", refill_cache: bool = False,
                  do_sample: bool = False, temperature: float = 1.0, top_p: float = 1.0, top_k: int = 0,
                  num_return_sequences: int = 1, generator: Optional[torch.Generator] = None):
    """Returns (ids [B, 1 + max_new_tokens] int64 incl. BOS, lengths [B] int64): row b's caption is
    ids[b, 1:lengths[b]] (EOS excluded); positions from lengths[b] on are what the lock-step loop kept
    generating and are to be ignored. `use_graphs` replays one captured CUDA graph of the bridge per
    prefix length (`DecodeStepGraphs`; pass `step_graphs` to reuse graphs captured for the same cache).
    `cache_positions` keeps block 0's cross-attention rows per text position in the cache (valid because
    `embed_fn` is a per-token lookup: the prefix rows do not change when a token is appended); pass
    False for an `embed_fn` that mixes positions.

    `precision="fp32"` runs the bridge with fp32 operands (csrc/exact_fp32.cu): the reference's own decode
    numerics (generate_caption runs without autocast, full_model.py:221-261), for which the token ids equal
    the fp32 reference's on every step; "bf16" is the tensor-core path (the reference's autocast numerics).
    `refill_cache=True` with a `kv_cache` from an earlier call recomputes that cache in place for
    `vision_features` (same shape), so `step_graphs` captured over it are replayed for new images.

    `do_sample=True` draws each token instead of taking the argmax (generate_caption(do_sample=True)): per row,
    the NaN / Inf guards above, z = logits / `temperature` (finite, > 0), the top-p nucleus (tokens whose
    strictly-larger-z softmax mass is < `top_p`, top_p in (0, 1]; ties at the threshold are kept together), and
    an exact draw from the renormalised nucleus (Gumbel-max over Philox4x32-10 of (seed, row, step); the rule is
    stated in include/b200_bridge.h). One 64-bit seed per call is drawn on the device from `generator` (a CUDA
    generator on the images' device; None = that device's default generator), so the loop never waits for the
    host and the same generator state gives the same captions. The step graphs still capture only the bridge;
    the sampler runs after each replay. `top_k` > 0 keeps, before the nucleus, only the tokens whose z is at least
    the top_k-th largest (ties kept together; 0 = off), as generate(do_sample=True, top_k=...) applies it between
    temperature and top-p.

    `num_return_sequences` = N > 1 (do_sample=True only, N <= 8) draws N captions per image over ONE cache of the
    images (`VisionKVCache(..., beams=N)`: each image's K/V is read once per step for all its N rows).
    `embed_fn` / `lm_fn` then see B*N rows in [B][N] order, and the results have B*N rows: row b*N + j is sample j
    of image b (the order of Hugging Face's repeat_interleave), drawn with the noise of row b*N + j of a sampled
    decode over `vision_features.repeat_interleave(N, 0)`. A `kv_cache` passed in must be built with beams=N.

    Bad `temperature` / `top_p` / `top_k` values, a `num_return_sequences` outside [1, 8] or above 1 without
    do_sample=True or use_cache=True, or a generator on another device raise ValueError before any kernel runs."""
    was_training = bridge.training
    bridge.eval()
    try:
        B = vision_features.shape[0]
        dev = vision_features.device
        if isinstance(num_return_sequences, bool) or not isinstance(num_return_sequences, numbers.Integral):
            raise ValueError(f"num_return_sequences must be an int, got {num_return_sequences!r}")
        N = int(num_return_sequences)
        if not 1 <= N <= 8:
            raise ValueError(f"num_return_sequences must be in [1, 8], got {N}")
        if N > 1 and not do_sample:
            raise ValueError("num_return_sequences > 1 needs do_sample=True (use beam_search_decode for the N best beams)")
        if N > 1 and not use_cache:
            raise ValueError("num_return_sequences > 1 shares one VisionKVCache per image: use_cache must stay True")
        if do_sample:
            temperature, top_p = float(temperature), float(top_p)
            if not (math.isfinite(temperature) and temperature > 0.0):
                raise ValueError(f"temperature must be finite and > 0, got {temperature}")
            if not (0.0 < top_p <= 1.0):
                raise ValueError(f"top_p must be in (0, 1], got {top_p}")
            if isinstance(top_k, bool) or not isinstance(top_k, numbers.Integral) or top_k < 0:
                raise ValueError(f"top_k must be an int >= 0, got {top_k!r}")
            if dev.type != "cuda":
                raise ValueError("do_sample=True needs the images on a CUDA device")
            gdev = None if generator is None else torch.device(generator.device)
            if gdev is not None and gdev.type == "cuda" and gdev.index is None:
                gdev = torch.device("cuda", torch.cuda.current_device())
            if gdev is not None and gdev != dev:
                raise ValueError(f"generator is on {generator.device}, the images on {dev}")
        kv_cache, step_graphs = _decode_setup(bridge, vision_features, max_new_tokens, kv_cache, use_cache, step_graphs,
                                              use_graphs, precision, refill_cache, beams=N)
        B *= N   # rows: N per image, [B][N]
        ids = torch.empty((B, 1 + max_new_tokens), dtype=torch.long, device=dev)
        ids[:, 0] = bos_token_id
        if do_sample:
            seed = torch.empty(1, dtype=torch.int64, device=dev).random_(generator=generator)
        for step in range(max_new_tokens):
            prefix = ids[:, :step + 1]
            kpos = step if (cache_positions and use_cache) else None
            if step_graphs is not None:
                hidden = step_graphs(embed_fn(prefix), cached_positions=kpos)
            else:
                hidden = bridge(vision_features, embed_fn(prefix), kv_cache=kv_cache if use_cache else None,
                                cached_positions=kpos)
            logits = lm_fn(hidden)
            if logits.dim() == 3:
                logits = logits[:, -1, :]
            if do_sample:
                if logits.dtype not in (torch.float32, torch.bfloat16) or logits.stride(-1) != 1:
                    logits = logits.float().contiguous()
                ops.sample_tokens(logits, temperature=temperature, top_p=top_p, top_k=int(top_k), seed=seed, step=step,
                                  out=ids[:, step + 1])
                continue
            logits = logits.float()
            # numerical guards of the reference, as tensor ops (no host sync)
            # (per row: the reference applies them to one caption at a time, full_model.py:270-283)
            bad = torch.isnan(logits).any(dim=-1, keepdim=True)
            logits = torch.where(bad, torch.zeros_like(logits), logits)
            logits = torch.where(torch.isinf(logits).any(dim=-1, keepdim=True), logits.clamp(min=-100, max=100), logits)
            ids[:, step + 1] = torch.argmax(logits, dim=-1)
        if eos_token_id is None:
            lengths = torch.full((B,), 1 + max_new_tokens, dtype=torch.long, device=dev)
        else:
            is_eos = ids[:, 1:] == eos_token_id
            first = torch.where(is_eos.any(dim=1), is_eos.float().argmax(dim=1), torch.full((B,), max_new_tokens, device=dev))
            lengths = first + 1
        return ids, lengths
    finally:
        bridge.train(was_training)


@torch.no_grad()
def beam_search_decode(bridge, vision_features: torch.Tensor, embed_fn: Callable[[torch.Tensor], torch.Tensor],
                       lm_fn: Callable[[torch.Tensor], torch.Tensor], *, num_beams: int, bos_token_id: int,
                       eos_token_id: Optional[int] = None, max_new_tokens: int = 50, length_penalty: float = 1.0,
                       early_stopping: bool = False, kv_cache: Optional[VisionKVCache] = None,
                       step_graphs: Optional[DecodeStepGraphs] = None, use_graphs: bool = False,
                       precision: str = "bf16", refill_cache: bool = False, num_return_sequences: int = 1):
    """Beam search over B images with `num_beams` = K beams each (generate(num_beams=K) of the Hugging Face stack the
    language model comes from; the rule, including where it differs from Hugging Face, is stated in
    include/b200_bridge.h at b200b_beam_step). Returns (ids [B, 1 + max_new_tokens] int64 incl. BOS, lengths [B]
    int64, scores [B] fp32): image b's caption is ids[b, 1:lengths[b]] (EOS excluded, as in `greedy_decode`) and
    scores[b] its sum of log-probabilities divided by n ** length_penalty.

    The B*K beam rows share their image's K/V (`VisionKVCache(..., beams=K)`): the cross-attention reads each
    image's cache once for all its beams. `embed_fn` / `lm_fn` see B*K rows, [B][K] (as in `greedy_decode`).
    Each step runs the bridge on the beams' prefixes, then one fused beam step on the logits of their last
    positions (`ops.beam_step`: log-softmax, scores, top-2K, finished hypotheses, the new beams' ids), then
    reorders the cached position rows by the chosen parents; nothing waits for the host, eagerly or with step
    graphs (`use_graphs` / `step_graphs`, as in `greedy_decode`). All beams run `max_new_tokens` steps in lock-step:
    an image whose search is done keeps its result while its rows keep flowing through the bridge.
    `num_return_sequences` = N returns each image's N best hypotheses (generate(num_beams=K, num_return_sequences=N)):
    the outputs then have B*N rows, row b*N + j the j-th best of image b (scores non-increasing in j; j = 0 is the
    N = 1 result).
    `num_beams` outside [1, 8], `num_return_sequences` outside [1, num_beams], a non-finite `length_penalty`, a
    `kv_cache` built for another number of beams or a `precision` other than "bf16" / "fp32" raise ValueError before
    any kernel runs."""
    K = int(num_beams)
    if not 1 <= K <= 8:
        raise ValueError(f"num_beams must be in [1, 8], got {num_beams}")
    if isinstance(num_return_sequences, bool) or not isinstance(num_return_sequences, numbers.Integral) or \
            not 1 <= num_return_sequences <= K:
        raise ValueError(f"num_return_sequences must be an int in [1, num_beams = {K}], got {num_return_sequences!r}")
    length_penalty = float(length_penalty)
    if not math.isfinite(length_penalty):
        raise ValueError(f"length_penalty must be finite, got {length_penalty}")
    if int(max_new_tokens) < 1:
        raise ValueError(f"max_new_tokens must be >= 1, got {max_new_tokens}")
    was_training = bridge.training
    bridge.eval()
    try:
        kv_cache, step_graphs = _decode_setup(bridge, vision_features, max_new_tokens, kv_cache, True, step_graphs,
                                              use_graphs, precision, refill_cache, beams=K)
        B = vision_features.shape[0]
        dev = vision_features.device
        T = int(max_new_tokens)
        ids = torch.empty((B * K, 1 + T), dtype=torch.long, device=dev)
        ids[:, 0] = bos_token_id
        ids_next = torch.empty_like(ids)
        parents = torch.empty(B * K, dtype=torch.long, device=dev)
        state = ops.BeamState(B, K, 1 + T, dev)
        for step in range(T):
            prefix = ids[:, :step + 1]
            if step_graphs is not None:
                hidden = step_graphs(embed_fn(prefix), cached_positions=step)
            else:
                hidden = bridge(vision_features, embed_fn(prefix), kv_cache=kv_cache, cached_positions=step)
            logits = lm_fn(hidden)
            if logits.dim() == 3:
                logits = logits[:, -1, :]
            if logits.dtype not in (torch.float32, torch.bfloat16) or logits.stride(-1) != 1:
                logits = logits.float().contiguous()
            ops.beam_step(logits, ids, ids_next, parents, state, step=step, eos_token_id=eos_token_id,
                          length_penalty=length_penalty, early_stopping=early_stopping)
            kv_cache.reorder_beams(parents)
            ids, ids_next = ids_next, ids
        return ops.beam_finalize(ids, state, steps=T, eos_token_id=eos_token_id, length_penalty=length_penalty,
                                 num_return_sequences=int(num_return_sequences))
    finally:
        bridge.train(was_training)
