"""Beam search (csrc/beam.cu, ops.beam_step / beam_finalize, VisionKVCache(beams=K), beam_search_decode).

The rule (include/b200_bridge.h, b200b_beam_step) is implemented here twice on the host: `host_step`, float64 numpy
over each beam's first 2K + 1 candidates, and `naive_step`, Python lists over a full sort of all K * V candidates.
They are checked against each other on the CPU; the kernels are checked against `host_step` on the GPU.

Where the kernel may differ from the float64 host (EPS): the kernel computes lse = m + ln S in fp32 with S a sum of
ex2.approx terms. Each term carries a relative error below 2^-22 (ex2.approx) plus 2^-24 |z - m| from rounding its
argument (negligible for the terms that matter); each thread adds at most 176 terms and rescales its partial at most
once per 16 loaded values (<= 11 times, 2^-22 each); the tree over threads, warps and CTAs adds 13 more rescales and
adds. Together |dS| / S < 11 * 2^-22 + 13 * 2^-22 + 200 * 2^-24 < 1.9e-5, so |d lse| < 1.9e-5 + 2^-24 |lse|. Then
c = fl(s + fl(z - lse)) adds two roundings, at most 2^-24 (|z| + |lse| + |s|) each. EPS = 4e-5 + 2^-22 (|z| + |lse|
+ |s|) bounds |c_kernel - c_host| with a factor of two to spare; two candidates are ordered alike on both sides when
their host scores differ by more than 2 EPS. A normalised score c / N adds one more rounding. An image's decisions are
compared only where every comparison it makes (adjacent candidates among the first 2K + 1, each finished-set offer
against the entry it competes with, the done test) clears that margin; exact ties (equal z of one row) resolve by
index on both sides and count as decided. Every test reports how many images were decided and requires nearly all.
"""
from __future__ import annotations

import ctypes as C
import itertools
import math

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu
ERR_SHAPE, ERR_ARG, ERR_WORKSPACE = -1, -3, -6
SENT = -7777
EPS0 = 4e-5
EPS_REL = 2.0 ** -22


# --------------------------------------------------------------------------------------------------------------------
# host references
# --------------------------------------------------------------------------------------------------------------------
def guard(x: np.ndarray) -> np.ndarray:
    """float32 [rows, V] -> float64: a row with a NaN -> zeros; else a row with an Inf -> clamped to [-100, 100]."""
    x = x.astype(np.float64)
    nan = np.isnan(x).any(1)
    x[nan] = 0.0
    inf = np.isinf(x).any(1) & ~nan
    x[inf] = np.clip(x[inf], -100.0, 100.0)
    return x


def lse_of(z: np.ndarray) -> float:
    m = z.max()
    return float(m + np.log(np.exp(z - m).sum()))


def top_of_row(z: np.ndarray, n: int) -> np.ndarray:
    """indices of the first n of a row by (z desc, index asc)"""
    if n >= len(z):
        idx = np.arange(len(z))
    else:
        thr = np.partition(z, len(z) - n)[len(z) - n]
        idx = np.nonzero(z >= thr)[0]
    return idx[np.lexsort((idx, -z[idx]))][:n]


def norm_den(n: int, alpha: float) -> float:
    return float(min(max(np.float32(n) ** np.float32(alpha), np.finfo(np.float32).tiny), np.finfo(np.float32).max))


class Image:
    """One image's beam state on the host: running scores s[K]; finished slots (score, len, seq, src) in slot order."""

    def __init__(self, K, s=None, hyps=None, count=0, done=False):
        self.K = K
        self.s = np.array([0.0] + [-np.inf] * (K - 1)) if s is None else np.asarray(s, np.float64)
        self.hyps = [] if hyps is None else [list(h) for h in hyps]   # [score, len, seq, src]
        self.count, self.done = count, done

    def offer(self, score, length, src, margin=0.0):
        """the finished-set rule; returns (slot or -1, decided)"""
        K = self.K
        if len(self.hyps) < K:
            self.hyps.append([score, length, self.count, src])
            self.count += 1
            return len(self.hyps) - 1, True
        w = min(range(K), key=lambda j: (self.hyps[j][0], self.hyps[j][2]))
        decided = abs(score - self.hyps[w][0]) > margin or score == self.hyps[w][0] == -np.inf
        if not score > self.hyps[w][0]:
            return -1, decided
        self.hyps[w] = [score, length, self.count, src]
        self.count += 1
        return w, decided


def host_step(img: Image, z: np.ndarray, eos: int, alpha: float, early: bool, t: int, zerr=None):
    """One step of the rule for one image (z: guarded float64 [K, V]). Mutates img; returns (parents, tokens,
    decided). Offers record src = ('beam', parent). zerr [K]: a bound on the error of the logits themselves (when
    they come from another implementation than the ones the kernel reads), added twice (z and lse) to EPS."""
    K, V = z.shape
    zerr = np.zeros(K) if zerr is None else zerr
    if img.done:
        pad = eos if eos >= 0 else 0
        return list(range(K)), [pad] * K, True
    cands = []
    for k in range(K):
        lse = lse_of(z[k])
        for v in top_of_row(z[k], 2 * K + 1):
            c = img.s[k] + (z[k, v] - lse)
            eps = (EPS0 + EPS_REL * (abs(z[k, v]) + abs(lse) + (abs(img.s[k]) if np.isfinite(img.s[k]) else 0.0))
                   + 2 * zerr[k] * (t + 1))
            cands.append((c, z[k, v], k * V + v, k, int(v), eps, lse))
    cands.sort(key=lambda e: (-e[0], -e[1], e[2]))
    decided = True
    for a, b in zip(cands[:2 * K], cands[1:2 * K + 1]):
        if a[0] == b[0] == -np.inf:
            continue
        exact = a[3] == b[3] and a[1] == b[1]            # the same row, equal z: an exact tie on both sides
        if not exact and abs(a[0] - b[0]) <= a[5] + b[5]:
            decided = False
    den = norm_den(t + 1, alpha)
    parents, tokens, news = [], [], []
    for r, (c, zz, f, k, v, eps, _) in enumerate(cands[:2 * K]):
        if len(parents) == K:
            break
        if v == eos:
            if r < K:
                sc = c / den
                _, ok = img.offer(sc, t + 1, ("beam", k), margin=2 * eps / den + 2 * EPS_REL * abs(sc))
                decided &= ok
            continue
        parents.append(k)
        tokens.append(v)
        news.append(c)
    assert len(parents) == K
    if len(img.hyps) >= K:
        if early:
            img.done = True
        else:
            worst = min(h[0] for h in img.hyps)
            best = max(news) / den
            if np.isfinite(best) and abs(worst - best) <= 2 * (EPS0 + EPS_REL * abs(best)) * max(1.0, 1.0 / den):
                decided = False
            img.done = bool(worst >= best)
    img.s = np.array(news)
    return parents, tokens, decided


def host_finalize(img: Image, steps: int, alpha: float):
    """(src, len, score) of the result; src = ('hyp', slot) or ('beam', k)"""
    hyps = [list(h[:3]) + [("hyp", j)] for j, h in enumerate(img.hyps)]
    tmp = Image(img.K, img.s, hyps, img.count, img.done)
    if not img.done:
        den = norm_den(steps, alpha)
        for k in range(img.K):
            tmp.offer(img.s[k] / den, steps + 1, ("beam", k))
    best = max(range(len(tmp.hyps)), key=lambda j: (tmp.hyps[j][0], -tmp.hyps[j][2]))
    h = tmp.hyps[best]
    return h[3], h[1], h[0]


def naive_step(s, hyps, count, z, eos, alpha, early, t):
    """The rule written out with Python lists: every one of the K * V candidates, fully sorted."""
    K, V = len(s), len(z[0])
    cand = []
    for k in range(K):
        m = max(z[k])
        lse = m + math.log(sum(math.exp(x - m) for x in z[k]))
        for v in range(V):
            cand.append((s[k] + (z[k][v] - lse), z[k][v], k * V + v, k, v))
    cand.sort(key=lambda e: (-e[0], -e[1], e[2]))
    n = t + 1
    den = float(n) ** alpha
    hyps = [list(h) for h in hyps]
    out_p, out_t, out_s = [], [], []
    for r, (c, _, _, k, v) in enumerate(cand[:2 * K]):
        if len(out_p) == K:
            break
        if v == eos:
            if r < K:
                if len(hyps) < K:
                    hyps.append([c / den, n, count])
                    count += 1
                else:
                    w = sorted(range(K), key=lambda j: (hyps[j][0], hyps[j][2]))[0]
                    if c / den > hyps[w][0]:
                        hyps[w] = [c / den, n, count]
                        count += 1
            continue
        out_p.append(k)
        out_t.append(v)
        out_s.append(c)
    done = len(hyps) >= K and (early or min(h[0] for h in hyps) >= max(out_s) / den)
    return out_p, out_t, out_s, hyps, count, done


# --------------------------------------------------------------------------------------------------------------------
# CPU tests
# --------------------------------------------------------------------------------------------------------------------
def test_host_step_equals_naive_full_sort():
    rng = np.random.default_rng(11)
    n = evictions = eos_low = eos_high = 0
    for case in range(240):
        K = int(rng.integers(1, 5))
        V = int(rng.integers(2, 9))
        eos = int(rng.integers(-1, V))
        alpha = [0.0, 1.0, 2.0][case % 3]
        early = bool(case % 2)
        t = int(rng.integers(0, 6))
        z = np.round(rng.standard_normal((K, V)) * 2, 1)        # rounded: exact ties inside rows
        if eos >= 0 and case % 4 == 0:
            z[:, eos] += 3.0                                        # EOS near the top of every beam
        s = np.sort(-rng.random(K) * 3)[::-1].copy()
        if case % 5 == 0:
            s[1:] = -np.inf
        nh = int(rng.integers(0, K + 1))
        hyps = [[float(-rng.random() * 3), int(rng.integers(1, 6)), j] for j in range(nh)]
        count = nh
        img = Image(K, s.copy(), [h + [("old", j)] for j, h in enumerate(hyps)], count)
        p, tk, decided = host_step(img, z, eos, alpha, early, t)
        wp, wt, ws, wh, wc, wd = naive_step(list(s), hyps, count, z.tolist(), eos, alpha, early, t)
        assert (p, tk) == (wp, wt), case
        assert np.allclose(img.s, ws)
        assert [h[:3] for h in img.hyps] == [h[:3] for h in wh] or np.allclose([h[0] for h in img.hyps],
                                                                             [h[0] for h in wh])
        assert img.count == wc and img.done == wd, case
        evictions += int(wc - count > len(wh) - nh)
        ranks = [i for i, (c, zz, f, k, v) in enumerate(sorted(
            [(s[k] + z[k, v] - lse_of(z[k]), z[k, v], k * V + v, k, v) for k in range(K) for v in range(V)],
            key=lambda e: (-e[0], -e[1], e[2]))[:2 * K]) if v == eos]
        eos_low += any(r < K for r in ranks)
        eos_high += any(r >= K for r in ranks)
        n += 1
    assert n == 240 and evictions > 5 and eos_low > 20 and eos_high > 10, (evictions, eos_low, eos_high)


def test_host_finalize_rule():
    img = Image(2, s=[-1.0, -3.0], hyps=[[-0.9, 3, 0, None]], count=1)
    src, ln, sc = host_finalize(img, 4, 1.0)
    # offers: beam 0 (-0.25) fills the set; beam 1 (-0.75) beats -0.9 and evicts it
    assert src == ("beam", 0) and ln == 5 and sc == -0.25
    img = Image(2, s=[-8.0, -9.0], hyps=[[-0.5, 3, 0, None], [-0.5, 4, 1, None]], count=2, done=True)
    assert host_finalize(img, 4, 1.0) == (("hyp", 0), 3, -0.5)         # done: no offers; a tie goes to the first


@pytest.fixture(scope="module")
def lib():
    from vlm_bridge_b200 import _lib, build

    h = C.CDLL(build.build())
    _lib._declare(h)
    return h


def _state_struct(addr, ld=8):
    from vlm_bridge_b200 import _lib

    return _lib.BeamState(addr, addr, addr, addr, addr, addr, addr, ld)


def test_beam_step_argument_codes_need_no_gpu(lib):
    """Every bad argument is rejected on the host before any CUDA call. Every call here fails a host check, so the
    dummy host pointers are never handed to a kernel (a call that passed them all would launch on a GPU machine);
    calls meant to show that an argument is accepted are given a workspace one byte short, the last check."""
    buf = C.create_string_buffer(64)
    a = C.addressof(buf)
    ws_ok = lib.b200b_beam_step_workspace_bytes(4, 3)
    assert ws_ok > 0
    assert lib.b200b_beam_step_workspace_bytes(0, 3) == 0 and lib.b200b_beam_step_workspace_bytes(4, 9) == 0
    ok = dict(logits=a, dtype=0, ld=16, batch=4, K=3, vocab=16, eos=1, alpha=1.0, early=0, step=2, ids=a, ids_next=a + 8,
              ld_ids=8, parents=a, state=_state_struct(a), ws=a, ws_bytes=ws_ok)

    def call(**kw):
        g = dict(ok, **kw)
        return lib.b200b_beam_step(g["logits"], g["dtype"], g["ld"], g["batch"], g["K"], g["vocab"], g["eos"],
                                   g["alpha"], g["early"], g["step"], g["ids"], g["ids_next"], g["ld_ids"], g["parents"],
                                   C.byref(g["state"]), g["ws"], g["ws_bytes"], None)

    for k in ("logits", "ids", "ids_next", "parents", "ws"):
        assert call(**{k: None}) == ERR_ARG and b"null" in lib.b200b_last_error()
    assert call(state=_state_struct(a).__class__(a, a, a, a, a, None, a, 8)) == ERR_ARG
    assert call(ids_next=a) == ERR_ARG                                      # ids == ids_next
    assert call(dtype=2) == ERR_ARG
    for K in (0, 9, -1):
        assert call(K=K) == ERR_ARG
    assert call(batch=0) == ERR_SHAPE
    assert call(vocab=1, ld=16, eos=0) == ERR_SHAPE
    for e in (-2, 16, 100):
        assert call(eos=e) == ERR_ARG
    assert call(eos=-1, ws_bytes=ws_ok - 1) == ERR_WORKSPACE                # eos = -1 (none) is accepted
    assert call(ld=15) == ERR_ARG
    assert call(step=-1) == ERR_ARG
    assert call(step=7) == ERR_ARG                                          # ld_ids = 8 < step + 2
    assert call(state=_state_struct(a, ld=3)) == ERR_ARG                    # ld_hyp < step + 2
    for al in (math.inf, -math.inf, math.nan):
        assert call(alpha=al) == ERR_ARG
    assert call(early=2) == ERR_ARG
    assert call(vocab=360449, ld=360449) == ERR_SHAPE                       # the sampler's vocabulary limit
    assert call(dtype=1, vocab=720897, ld=720897) == ERR_SHAPE
    ws8 = lib.b200b_beam_step_workspace_bytes(1, 8)
    assert call(K=8, vocab=300000, ld=300000, batch=1, ws_bytes=ws8 - 1) == ERR_WORKSPACE   # within the limit
    assert call(batch=1 << 27) == ERR_SHAPE                                 # rows * 8 beyond 2^31
    assert call(ws_bytes=ws_ok - 1) == ERR_WORKSPACE


def test_beam_finalize_argument_codes_need_no_gpu(lib):
    buf = C.create_string_buffer(64)
    a = C.addressof(buf)
    ok = dict(batch=2, K=3, eos=1, alpha=1.0, steps=4, ids=a, ld_ids=5, state=_state_struct(a), out=a, ld_out=5,
              out_len=a, out_score=a)

    def call(**kw):
        g = dict(ok, **kw)
        return lib.b200b_beam_finalize(g["batch"], g["K"], g["eos"], g["alpha"], g["steps"], g["ids"], g["ld_ids"],
                                       C.byref(g["state"]), g["out"], g["ld_out"], g["out_len"], g["out_score"], None)

    for k in ("ids", "out", "out_len", "out_score"):
        assert call(**{k: None}) == ERR_ARG
    assert call(K=0) == ERR_ARG and call(K=9) == ERR_ARG
    assert call(batch=0) == ERR_SHAPE and call(steps=0) == ERR_SHAPE
    assert call(eos=-2) == ERR_ARG
    assert call(ld_ids=4) == ERR_ARG and call(ld_out=4) == ERR_ARG
    assert call(state=_state_struct(a, ld=4)) == ERR_ARG
    assert call(alpha=math.nan) == ERR_ARG


def test_beam_search_decode_arguments_raise_value_error():
    import types

    from vlm_bridge_b200 import BridgeLite, VisionKVCache, beam_search_decode

    m = BridgeLite(vision_dim=32, language_dim=64, num_heads_cross=1, num_heads_self=1)
    v = torch.randn(1, 4, 32)
    fns = (lambda t: torch.zeros(t.shape + (64,)), lambda y: y[:, -1, :])
    for nb in (0, 9, -1):
        with pytest.raises(ValueError, match="num_beams"):
            beam_search_decode(m, v, *fns, num_beams=nb, bos_token_id=2)
    for lp in (math.inf, -math.inf, math.nan):
        with pytest.raises(ValueError, match="length_penalty"):
            beam_search_decode(m, v, *fns, num_beams=2, bos_token_id=2, length_penalty=lp)
    with pytest.raises(ValueError, match="precision"):
        beam_search_decode(m, v, *fns, num_beams=2, bos_token_id=2, precision="fp16")
    c = object.__new__(VisionKVCache)
    c.batch, c.len_vision, c.beams, c.precision = 1, 4, 3, "bf16"
    with pytest.raises(ValueError, match="beams=3"):
        beam_search_decode(m, v, *fns, num_beams=2, bos_token_id=2, kv_cache=c)
    assert m.training                                   # the mode is restored on the error path
    with pytest.raises(ValueError, match="beams"):
        VisionKVCache(types.SimpleNamespace(), torch.randn(1, 4, 32), beams=9)


def test_beam_cache_rejects_a_mismatched_text_batch_before_any_kernel():
    """A text batch other than images x beams would make the decode kernels address K/V past the cache: the
    forward raises before it builds any kernel dims (here on a CPU module, which would fail later otherwise)."""
    from vlm_bridge_b200 import BridgeLite, VisionKVCache

    m = BridgeLite(vision_dim=32, language_dim=64, num_heads_cross=1, num_heads_self=1).eval()
    c = object.__new__(VisionKVCache)
    c.batch, c.len_vision, c.beams, c.precision, c.max_positions, c.positions_filled = 2, 5, 3, "bf16", 8, 0
    c.x1 = torch.empty(6, 8, 64)
    c.kv = c.kv_packed = c.kv_tc = c.kv32 = None
    for rows in (2, 5, 7, 12):
        with torch.no_grad(), pytest.raises(RuntimeError, match="2 images x 3 beams"):
            m(None, torch.randn(rows, 1, 64), kv_cache=c)
        with pytest.raises(RuntimeError, match="2 images x 3 beams"):
            m._run_forward_beams(torch.randn(rows, 1, 64), c)
    c.precision = "fp32"
    with torch.no_grad(), pytest.raises(RuntimeError, match="2 images x 3 beams"):
        m(None, torch.randn(2, 1, 64), kv_cache=c)
    with torch.no_grad(), pytest.raises(RuntimeError, match="CUDA"):
        m(None, torch.randn(6, 1, 64), kv_cache=c)          # the right batch passes the check


def test_reorder_beams_gathers_filled_rows_in_place():
    from vlm_bridge_b200 import VisionKVCache

    c = object.__new__(VisionKVCache)
    c.batch, c.beams, c.positions_filled = 2, 3, 2
    c.x1 = torch.arange(6 * 4 * 2, dtype=torch.float32).view(6, 4, 2)
    before, ptr = c.x1.clone(), c.x1.data_ptr()
    parents = torch.tensor([2, 2, 0, 3, 5, 4])
    c.reorder_beams(parents)
    assert c.x1.data_ptr() == ptr
    assert torch.equal(c.x1[:, :2], before[parents, :2]) and torch.equal(c.x1[:, 2:], before[:, 2:])
    with pytest.raises(RuntimeError, match="parents"):
        c.reorder_beams(torch.tensor([0, 1, 2]))


# --------------------------------------------------------------------------------------------------------------------
# GPU, op level
# --------------------------------------------------------------------------------------------------------------------
def _make_case(B, K, V, dtype, case):
    """logits [B*K, V] (float32 values, representable in dtype), a mid-search state and prefixes"""
    g = np.random.default_rng(1000 + case)
    R = B * K
    x = (g.standard_normal((R, V)) * 3.0).astype(np.float32)
    if V >= 8:
        x[1::2] = np.round(x[1::2] * 4) / 4                 # ties
    eos = int(g.integers(0, V)) if case % 3 else -1
    if eos >= 0:
        boost = g.choice([-0.5, 0.2, 1.0, 3.0], size=R)
        x[:, eos] = x.max(1) + boost
    if V >= 4 * K + 4:                                      # exact duplicates straddling the 2K boundary of row 0
        o = np.argsort(-x[0], kind="stable")
        x[0, o[2 * K]] = x[0, o[2 * K - 1]]
        x[0, o[2 * K + 1]] = x[0, o[2 * K - 1]]
    if R >= 3:
        x[1, V // 2] = np.inf
        x[2, (2 * V) // 3] = np.nan
    tdt = torch.float32 if dtype == "f32" else torch.bfloat16
    x = torch.from_numpy(x).to(tdt).float().numpy()          # the values the kernel sees
    t = 0 if case % 4 == 0 else int(g.integers(1, 7))
    s = np.full(R, -np.inf, np.float32)
    s[::K] = 0.0
    if t > 0:
        s = np.sort(-(g.random(R) * 6).astype(np.float32).reshape(B, K), axis=1)[:, ::-1].reshape(R).copy()
        if case % 5 == 1 and K > 1:
            s[K - 1::K] = -np.inf
    count = np.zeros(B, np.int32)
    hs = np.full(R, -np.inf, np.float32)
    hl = np.zeros(R, np.int32)
    hq = np.zeros(R, np.int32)
    done = np.zeros(B, np.int32)
    if t > 0:
        for b in range(B):
            nh = int(g.integers(0, K + 1))
            count[b] = nh + int(g.integers(0, 3)) if nh == K else nh
            hs[b * K:b * K + nh] = -(g.random(nh) * 3).astype(np.float32)
            hl[b * K:b * K + nh] = g.integers(1, t + 1, nh)
            hq[b * K:b * K + nh] = np.arange(nh)
        if B > 1:
            done[B - 1] = 1                                 # a frozen image
            count[B - 1] = max(count[B - 1], 1)
    ids = g.integers(0, V, (R, t + 1)).astype(np.int64)
    ids[:, 0] = 2 % V
    return x, eos, t, s, (hs, hl, hq, count, done), ids


def _run_op_case(B, K, V, dtype, case, alpha, early):
    from vlm_bridge_b200 import ops

    x, eos, t, s, (hs, hl, hq, count, done), ids_np = _make_case(B, K, V, dtype, case)
    R = B * K
    tdt = torch.float32 if dtype == "f32" else torch.bfloat16
    pad = 8 if case % 2 == 0 else 13
    buf = torch.full((R, V + pad), math.nan, dtype=tdt, device="cuda")
    buf[:, :V] = torch.from_numpy(x).to(tdt).cuda()
    L = t + 2 + 3                                                        # room beyond t + 1: must stay untouched
    ids = torch.full((R, L), SENT, dtype=torch.int64, device="cuda")
    ids[:, :t + 1] = torch.from_numpy(ids_np).cuda()
    ids_next = torch.full((R, L), SENT, dtype=torch.int64, device="cuda")
    pbuf = torch.full((R + 5,), SENT, dtype=torch.int64, device="cuda")
    parents = pbuf[2:2 + R]
    st = ops.BeamState(B, K, L, "cuda")
    st.beam_scores.copy_(torch.from_numpy(s))
    st.hyp_scores.copy_(torch.from_numpy(hs))
    st.hyp_lens.copy_(torch.from_numpy(hl))
    st.hyp_seq.copy_(torch.from_numpy(hq))
    st.hyp_count.copy_(torch.from_numpy(count))
    st.done.copy_(torch.from_numpy(done))
    st.hyp_ids.fill_(SENT)
    before = {k: getattr(st, k).cpu() for k in ("beam_scores", "hyp_scores", "hyp_lens", "hyp_seq", "hyp_count",
                                                  "done", "hyp_ids")}
    ops.beam_step(buf[:, :V], ids, ids_next, parents, st, step=t, eos_token_id=None if eos < 0 else eos,
                  length_penalty=alpha, early_stopping=early)
    torch.cuda.synchronize()
    pb = pbuf.cpu()
    assert (pb[:2] == SENT).all() and (pb[2 + R:] == SENT).all(), "a write outside parents"
    nxt = ids_next.cpu().numpy()
    assert (nxt[:, t + 2:] == SENT).all(), "a write beyond position t + 1"
    got = {k: getattr(st, k).cpu() for k in before}
    zg = guard(x)
    decided = 0
    for b in range(B):
        rows = slice(b * K, (b + 1) * K)
        hyps = [[float(hs[b * K + j]), int(hl[b * K + j]), int(hq[b * K + j]), ("old", j)]
                for j in range(min(int(count[b]), K))]
        img = Image(K, s[rows].astype(np.float64), hyps, int(count[b]), bool(done[b]))
        par, tok, ok = host_step(img, zg[rows], eos, alpha, early, t)
        if done[b]:
            for k in before:
                if k != "hyp_ids":
                    kk = slice(b, b + 1) if k in ("hyp_count", "done") else rows
                    assert torch.equal(got[k][kk], before[k][kk]), (k, b)
            assert torch.equal(got["hyp_ids"][rows], before["hyp_ids"][rows])
        if not ok:
            continue
        decided += 1
        assert list(pb[2 + b * K:2 + (b + 1) * K].numpy() - b * K) == par, (B, K, V, dtype, case, b)
        assert list(nxt[rows, t + 1]) == tok, (B, K, V, dtype, case, b)
        for k in range(K):
            assert (nxt[b * K + k, :t + 1] == ids_np[b * K + par[k], :t + 1]).all()
        if not done[b]:
            ns = got["beam_scores"][rows].numpy().astype(np.float64)
            fin = np.isfinite(img.s)
            assert (np.isfinite(ns) == fin).all() and np.allclose(ns[fin], img.s[fin], rtol=0, atol=1e-4)
            assert int(got["hyp_count"][b]) == img.count and int(got["done"][b]) == int(img.done)
            for j, h in enumerate(img.hyps):
                gs = float(got["hyp_scores"][b * K + j])
                assert gs == h[0] or abs(gs - h[0]) <= 1e-4 * max(1.0, abs(h[0])), (b, j, gs, h[0])
                assert int(got["hyp_lens"][b * K + j]) == h[1] and int(got["hyp_seq"][b * K + j]) == h[2]
                hrow = got["hyp_ids"][b * K + j].numpy()
                if h[3][0] == "beam":                       # added this step: the parent's prefix and the EOS
                    assert (hrow[:t + 1] == ids_np[b * K + h[3][1], :t + 1]).all() and hrow[t + 1] == eos
                else:
                    assert (hrow == SENT).all()
    return decided, B


OP_KS = (1, 2, 3, 4, 8)
OP_BS = (1, 3, 32)


def _op_grid(V, dtype):
    if V <= 4096:
        return [(b, k) for k in OP_KS for b in OP_BS]
    off = 0 if dtype == "f32" else 1
    return [(OP_BS[(j + off) % 3], k) for j, k in enumerate(OP_KS)]


@gpu
@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("V", [2, 17, 4096, 256000, 256001])
def test_beam_step_against_host_reference(dtype, V):
    decided = total = 0
    for case, (B, K) in enumerate(_op_grid(V, dtype)):
        alpha = (0.0, 1.0, 2.0)[case % 3]
        d, n = _run_op_case(B, K, V, dtype, case, alpha, bool(case % 2))
        decided += d
        total += n
    print(f"beam_step {dtype} V={V}: {decided} / {total} images decided and equal")
    assert decided >= 0.95 * total


@gpu
def test_beam_step_k1_is_the_greedy_argmax():
    from vlm_bridge_b200 import ops

    for V, dt in ((17, torch.float32), (32000, torch.bfloat16), (256000, torch.float32)):
        B = 40
        g = torch.Generator().manual_seed(V)
        x = torch.randn(B, V, generator=g) * 3.0
        x[1, 5] = math.inf
        x[2, 7] = math.nan
        xd = x.to(dt).cuda()
        st = ops.BeamState(B, 1, 4, "cuda")
        ids = torch.full((B, 4), 2, dtype=torch.int64, device="cuda")
        nxt = torch.empty_like(ids)
        par = torch.empty(B, dtype=torch.int64, device="cuda")
        ops.beam_step(xd, ids, nxt, par, st, step=0, eos_token_id=None)
        lf = xd.float()
        lf = torch.where(torch.isnan(lf).any(-1, keepdim=True), torch.zeros_like(lf), lf)
        lf = torch.where(torch.isinf(lf).any(-1, keepdim=True), lf.clamp(-100, 100), lf)
        assert torch.equal(nxt[:, 1], torch.argmax(lf, dim=-1)), V
        assert torch.equal(par, torch.arange(B, device="cuda"))


@gpu
def test_beam_step_tolerates_a_corrupt_state_and_checks_shapes():
    """A NaN running score (which reset() never writes) ranks last like -inf, and a negative hyp_count counts as 0:
    parents stay inside their image. The wrapper rejects ids views too narrow for position step + 1."""
    from vlm_bridge_b200 import ops

    B, K, V, t = 3, 4, 4096, 2
    g = torch.Generator().manual_seed(9)
    x = (torch.randn(B * K, V, generator=g) * 3).cuda()
    st = ops.BeamState(B, K, 8, "cuda")
    st.beam_scores.copy_(torch.tensor([-1.0, math.nan, -2.0, -3.0] * B))
    st.hyp_count.copy_(torch.tensor([-5, 0, 2], dtype=torch.int32))
    st.hyp_scores.fill_(-1.0)
    ids = torch.randint(0, V, (B * K, 8), generator=g).cuda()
    nxt = torch.empty_like(ids)
    par = torch.empty(B * K, dtype=torch.int64, device="cuda")
    ops.beam_step(x, ids, nxt, par, st, step=t, eos_token_id=1)
    p = par.cpu().view(B, K)
    assert bool(((p >= torch.arange(B)[:, None] * K) & (p < torch.arange(1, B + 1)[:, None] * K)).all())
    assert not bool((p % K == 1).any())                  # the NaN beam is never a parent
    assert bool(torch.isfinite(st.beam_scores).all())
    with pytest.raises(RuntimeError, match="columns"):
        ops.beam_step(x, ids[:, :t + 1], nxt[:, :t + 1], par, st, step=t, eos_token_id=1)


# --------------------------------------------------------------------------------------------------------------------
# GPU, the bridge forward over a beam cache
# --------------------------------------------------------------------------------------------------------------------
def _bridge(seed=0):
    from oracle import bridge_oracle as O
    from vlm_bridge_b200 import BridgeLite

    m = BridgeLite(dropout=0.0)
    m.load_state_dict(O.init_state_dict(seed), strict=True)
    return m.cuda().eval()


@gpu
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("K,s", [(3, 1), (4, 5), (8, 9), (2, 40)])
def test_beam_forward_equals_replicated_cache(precision, K, s):
    """The beam layout (one query block of K*s rows per image) against a cache of the images repeated K times.
    Equal bits where both sides run the same cross-attention kernel family (fp32; bf16: the mma.sync decode kernel
    up to 32 query rows, the tcgen05 one for 33..64, the projection-output path beyond), else within 5e-3 of the
    output maximum, the bound test_decode_gpu uses across those families."""
    from vlm_bridge_b200 import VisionKVCache
    from vlm_bridge_b200.bridge import TC_DECODE_MIN_LEN

    m = _bridge()
    g = torch.Generator().manual_seed(50 + K * 10 + s)
    B, Nv = 2, 257
    vision = torch.randn(B, Nv, 1024, generator=g).cuda()
    text = torch.randn(B * K, s, 2304, generator=g).cuda()
    with torch.no_grad():
        beam = VisionKVCache(m, vision, precision=precision, beams=K)
        rep = VisionKVCache(m, vision.repeat_interleave(K, 0), precision=precision)
        yb, yr = m(None, text, kv_cache=beam), m(None, text, kv_cache=rep)

        def family(rows):
            if precision == "fp32":
                return "fp32"
            return "packed" if rows < TC_DECODE_MIN_LEN else ("tc" if rows <= 64 else "kv")

        def check(a, b, same, what):
            rel = float((a - b).abs().max() / b.abs().max())
            print(f"{precision} K={K} s={s} {what}: same kernel family {same}, equal={torch.equal(a, b)}, rel={rel:.2e}")
            assert torch.equal(a, b) if same else rel <= 5e-3, (what, rel)

        check(yb, yr, family(K * s) == family(s), "full prefix")
        # cached positions: grow the prefix one token at a time on both caches
        for j in range(1, s + 1):
            yb = m(None, text[:, :j], kv_cache=beam, cached_positions=j - 1)
            yr = m(None, text[:, :j], kv_cache=rep, cached_positions=j - 1)
        # block 0's cross-attention ran over K vs 1 new rows per image, the later blocks' over K*s vs s
        check(yb, yr, family(K) == family(1) and family(K * s) == family(s), "cached positions")
        if s >= 2:
            # reorder_beams, then a cached step, against a full recompute of the reordered prefixes
            par = torch.arange(B * K, device="cuda").view(B, K).flip(1).reshape(-1)
            beam.reorder_beams(par)
            t2 = torch.cat([text[par, :s], text[:, :1]], dim=1)
            y_inc = m(None, t2, kv_cache=beam, cached_positions=s)
            y_full = m(None, t2, kv_cache=beam)
            assert float((y_inc - y_full).abs().max() / y_full.abs().max()) <= 5e-3


# --------------------------------------------------------------------------------------------------------------------
# GPU, end to end
# --------------------------------------------------------------------------------------------------------------------
E2E_B, E2E_K, E2E_NV, E2E_STEPS, E2E_V = 2, 3, 33, 8, 512


def _e2e(V=E2E_V, B=E2E_B, nv=E2E_NV, seed=20):
    from oracle import bridge_oracle as O

    sd = O.init_state_dict(1)
    g = torch.Generator().manual_seed(seed)
    vision = torch.randn(B, nv, 1024, generator=g)
    embed = torch.randn(V, 2304, generator=g)
    head = torch.randn(V, 2304, generator=g) / 48.0
    m = _bridge(1)
    ed, hd = embed.cuda(), head.cuda()
    return sd, vision, embed, head, m, (lambda t: ed[t]), (lambda y: y[:, -1, :] @ hd.t())


@gpu
def test_beam_search_fp32_matches_host_beam_search_over_the_oracle():
    """beam_search_decode(precision="fp32") against the rule run in float64 on the fp32 CPU oracle's logits of the
    same prefixes (teacher forcing). The fp32 CUDA logits differ from the oracle's by less than 1e-5 of their maximum
    (asserted in test_decode_c4_gpu); that bound joins EPS, once per step since it accumulates in the beam scores.
    An image is compared if every decision it made cleared the margin; the bound is conservative (it lets the logit error add up over every step), so about
    half of the 32 images (4 images, 4 decoding settings, 2 images each) are compared."""
    from oracle import bridge_oracle as O
    from vlm_bridge_b200 import beam_search_decode

    B, K, T = E2E_B, E2E_K, E2E_STEPS
    compared = total = 0
    loaded = None
    for seed, (eos, alpha, early) in itertools.product((20, 21, 22, 23), ((1, 1.0, False), (7, 0.0, True),
                                                                          (None, 2.0, False), (3, 1.0, True))):
        if loaded != seed:                 # new images (and read-out) per seed, same bridge weights
            sd, vision, embed, head, m, ef, lf = _e2e(seed=seed)
            loaded = seed
        ids, lengths, scores = beam_search_decode(m, vision.cuda(), ef, lf, num_beams=K, bos_token_id=2,
                                                  eos_token_id=eos, max_new_tokens=T, length_penalty=alpha,
                                                  early_stopping=early, precision="fp32")
        ids, lengths, scores = ids.cpu(), lengths.cpu(), scores.cpu()
        kvs = [(k.repeat_interleave(K, 0), v.repeat_interleave(K, 0)) for k, v in O.vision_kv(sd, vision)]
        e = -1 if eos is None else eos
        imgs = [Image(K) for _ in range(B)]
        prefix = [[[2] for _ in range(K)] for _ in range(B)]
        hyp_ids = [dict() for _ in range(B)]
        ok = [True] * B
        for t in range(T):
            rows = torch.tensor([prefix[b][k] for b in range(B) for k in range(K)])
            y = O.bridge_forward_cached(sd, kvs, embed[rows])
            z = guard((y[:, -1, :] @ head.t()).numpy().astype(np.float32))
            for b in range(B):
                old = [list(p) for p in prefix[b]]
                zb = z[b * K:(b + 1) * K]
                par, tok, dec = host_step(imgs[b], zb, e, alpha, early, t, zerr=1e-5 * np.abs(zb).max(1))
                ok[b] &= dec
                for h in imgs[b].hyps:
                    if h[3][0] == "beam":                       # added this step
                        hyp_ids[b][h[2]] = old[h[3][1]] + [e]
                        h[3] = ("seq", h[2])
                prefix[b] = [old[par[k]] + [tok[k]] for k in range(K)]
        for b in range(B):
            total += 1
            if not ok[b]:
                continue
            compared += 1
            src, ln, sc = host_finalize(imgs[b], T, alpha)
            want = prefix[b][src[1]] if src[0] == "beam" else hyp_ids[b][imgs[b].hyps[src[1]][2]]
            assert int(lengths[b]) == ln, (eos, b)
            assert ids[b, :ln].tolist() == want[:ln], (eos, b)
            assert abs(float(scores[b]) - sc) <= 1e-3 * max(1.0, abs(sc)), (eos, b, float(scores[b]), sc)
    print(f"beam_search_decode fp32 vs oracle: {compared} / {total} images decided and equal")
    assert compared >= 12                  # seeded: the same images clear the margin on every run


@gpu
def test_beam_search_k1_graphs_sync_free_and_refill():
    from vlm_bridge_b200 import VisionKVCache, beam_search_decode, greedy_decode
    from vlm_bridge_b200.decode import DecodeStepGraphs

    sd, vision, embed, head, m, ef, lf = _e2e(B=4)
    vc = vision.cuda()
    kw = dict(bos_token_id=2, max_new_tokens=E2E_STEPS)
    for precision in ("bf16", "fp32"):
        gi, _ = greedy_decode(m, vc, ef, lf, precision=precision, **kw)
        bi, bl, _ = beam_search_decode(m, vc, ef, lf, num_beams=1, precision=precision, **kw)
        assert torch.equal(gi, bi) and bool((bl == E2E_STEPS + 1).all()), precision
    K = 3
    cache = VisionKVCache(m, vc, beams=K)
    graphs = DecodeStepGraphs(m, cache)
    kw = dict(kw, eos_token_id=1, num_beams=K, kv_cache=cache)
    eager = beam_search_decode(m, vc, ef, lf, **kw)
    replay = beam_search_decode(m, vc, ef, lf, step_graphs=graphs, **kw)
    for a, b in zip(eager, replay):
        assert torch.equal(a, b)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        beam_search_decode(m, vc, ef, lf, **kw)
        beam_search_decode(m, vc, ef, lf, step_graphs=graphs, **kw)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    # new images through the same cache and graphs
    v2 = torch.randn_like(vc)
    ref = beam_search_decode(m, v2, ef, lf, num_beams=K, bos_token_id=2, eos_token_id=1, max_new_tokens=E2E_STEPS)
    got = beam_search_decode(m, v2, ef, lf, step_graphs=graphs, refill_cache=True, **kw)
    for a, b in zip(ref, got):
        assert torch.equal(a, b)


@gpu
@pytest.mark.timeout(1500)
def test_beam_search_c4_deterministic_and_scores_are_teacher_forced_log_probs():
    """C4 size (32 images, K = 4, 64 steps, 257 vision tokens, V = 256 000 stand-in read-out, graphs over a refilled
    cache): two bf16 runs give the same bits; in fp32 each score is the teacher-forced sum of log-probabilities of
    its caption (EOS included) through the same bridge, divided by n ** alpha (n counts the EOS)."""
    from vlm_bridge_b200 import VisionKVCache, beam_search_decode
    from vlm_bridge_b200.decode import DecodeStepGraphs

    B, K, T, V = 32, 4, 64, 256000
    g = torch.Generator(device="cuda").manual_seed(20)
    vision = torch.randn(B, 257, 1024, device="cuda", generator=g)
    embed = torch.randn(V, 2304, device="cuda", generator=g)
    head = torch.randn(V, 2304, device="cuda", generator=g) / 48.0
    m = _bridge(1)
    ef, lf = (lambda t: embed[t]), (lambda y: y[:, -1, :] @ head.t())
    cache = VisionKVCache(m, vision, max_positions=T, beams=K)
    graphs = DecodeStepGraphs(m, cache)
    kw = dict(num_beams=K, bos_token_id=2, eos_token_id=1, max_new_tokens=T, length_penalty=1.0)
    a = beam_search_decode(m, vision, ef, lf, kv_cache=cache, step_graphs=graphs, refill_cache=True, **kw)
    b = beam_search_decode(m, vision, ef, lf, kv_cache=cache, step_graphs=graphs, refill_cache=True, **kw)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    ids, lengths, scores = beam_search_decode(m, vision, ef, lf, precision="fp32", **kw)
    # n = tokens including the EOS (positions past a caption hold the EOS, so ids[b, n] is it when there is one)
    n = torch.where(lengths <= T, lengths, lengths - 1)
    total = torch.zeros(B, dtype=torch.float64, device="cuda")
    c32 = VisionKVCache(m, vision, max_positions=0, precision="fp32")
    with torch.no_grad():
        for j in range(T):              # prefix j + 1 -> the log-probability of token j + 1 (the self-attention
            y = m(None, embed[ids[:, :j + 1]], kv_cache=c32)        # is non-causal: one forward per prefix)
            logp = torch.log_softmax(y[:, -1, :] @ head.t(), dim=-1)
            lp = logp.gather(1, ids[:, j + 1:j + 2])[:, 0].double()
            total += torch.where(j < n, lp, torch.zeros_like(lp))
    want = total / n.double()
    err = (scores.double() - want).abs()
    print(f"C4 beam search: largest |score - teacher-forced score| = {float(err.max()):.2e}")
    assert bool((err <= 1e-3 * want.abs().clamp(min=1.0)).all()), (scores, want)
