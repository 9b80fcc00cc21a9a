"""Top-k in the fused sampler (b200b_sample_tokens_top_k, ops.sample_tokens(top_k=...)), the N best hypotheses of a beam
search (b200b_beam_finalize_top, ops.beam_finalize(num_return_sequences=N)) and several captions per image
(greedy_decode(do_sample=True, num_return_sequences=N), beam_search_decode(num_return_sequences=N)).

The sampling rule (include/b200_bridge.h) fixes every random number, so the kernel is checked token for token against a
float64 host sampler fed with the same Philox words. The host divides by the temperature in fp32 as the rule says, so
host and kernel see the same z values and the top-k threshold (a selection by count over those z) must agree exactly:
every kernel id must lie in the host's top-k set. The nucleus edge and the Gumbel keys use the tolerances of the top-p
sampler (DELTA on a mass ratio, EPS on a key, argued in test_sampling_gpu.py); a row is "decided" when no candidate
other than the host pick lies within them, and every decided row must be exact.

The finalize rule is checked in fp32 on the host: the finished scores are read back from the state and a running
beam's score s / n^alpha is one fp32 division (alpha in {0, 1, 2}, so n^alpha is exact), so the host ordering is exact.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu
TAG = 0x5A3B1E00
EPS_SCALE = 2.0 ** -20
DELTA = 1e-4
ERR_SHAPE, ERR_ARG = -1, -3
SENT = -7777
_MASK32 = np.uint64(0xFFFFFFFF)


# --------------------------------------------------------------------------------------------------------------------
# float64 host sampler with top-k
# --------------------------------------------------------------------------------------------------------------------
def philox4x32_10(ctr: np.ndarray, key) -> np.ndarray:
    """ctr uint32 [..., 4], key (k0, k1) -> uint32 [..., 4] (Salmon et al. 2011, 10 rounds)."""
    c0, c1, c2, c3 = (ctr[..., i].astype(np.uint64) for i in range(4))
    k0, k1 = np.uint64(int(key[0]) & 0xFFFFFFFF), np.uint64(int(key[1]) & 0xFFFFFFFF)
    m0, m1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    for _ in range(10):
        p0, p1 = m0 * c0, m1 * c2          # < 2^64: no wrap-around
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _MASK32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _MASK32
        k0 = (k0 + np.uint64(0x9E3779B9)) & _MASK32
        k1 = (k1 + np.uint64(0xBB67AE85)) & _MASK32
    return np.stack([c0, c1, c2, c3], -1).astype(np.uint32)


def host_words(idx: np.ndarray, row: int, step: int, seed: int) -> np.ndarray:
    """The 32-bit Philox word of each vocabulary index in idx (sorted int64) for (row, step, seed)."""
    groups, inv = np.unique(idx >> 2, return_inverse=True)
    ctr = np.empty((len(groups), 4), np.uint32)
    ctr[:, 0] = (groups & 0xFFFFFFFF).astype(np.uint32)
    ctr[:, 1] = row
    ctr[:, 2] = step & 0xFFFFFFFF
    ctr[:, 3] = TAG
    w = philox4x32_10(ctr, (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF))
    return w[inv, idx & 3]


def host_gumbel(w: np.ndarray) -> np.ndarray:
    """g = -ln(-ln u), u = ((w >> 8) + 0.5) 2^-24, exact in float64 (1 - u too)."""
    m = (w >> 8).astype(np.float64)
    u = (m + 0.5) * 2.0 ** -24
    nlu = np.where(m < 2 ** 23, -np.log(u), -np.log1p(-(1.0 - u)))
    return -np.log(nlu)


def host_guard(x: np.ndarray) -> np.ndarray:
    """x float32 [rows, V]: a row with a NaN -> zeros; else a row with an Inf -> clamped to [-100, 100]."""
    x = x.copy()
    nan = np.isnan(x).any(1)
    x[nan] = 0.0
    inf = np.isinf(x).any(1) & ~nan
    x[inf] = np.clip(x[inf], -100.0, 100.0)
    return x


def host_z(x_row: np.ndarray, temperature: float) -> np.ndarray:
    return (x_row.astype(np.float32) / np.float32(temperature)).astype(np.float32).astype(np.float64)


def topk_pass(z: np.ndarray, k: int) -> np.ndarray:
    """Rule 3a: z_i >= the k-th largest z (duplicates counted); everything for k == 0 or k >= V."""
    if k == 0 or k >= len(z):
        return np.ones(len(z), bool)
    return z >= np.partition(z, len(z) - k)[len(z) - k]


def mass_above(z: np.ndarray) -> np.ndarray:
    """softmax(z) mass of the tokens with strictly larger z, per token (float64)."""
    e = np.exp(z - z.max())
    order = np.argsort(-z, kind="stable")
    zs, es = z[order], e[order]
    excl = np.concatenate([[0.0], np.cumsum(es)[:-1]])
    start = np.concatenate([[True], zs[1:] != zs[:-1]])
    first = np.maximum.accumulate(np.where(start, np.arange(len(z)), 0))
    out = np.empty_like(z)
    out[order] = excl[first] / es.sum()
    return out


def host_sample(x_row, temperature, top_k, top_p, seed, step, row):
    """(host pick, candidate ids the kernel may return, top-k set) for one guarded float32 row."""
    z = host_z(x_row, temperature)
    passing = topk_pass(z, top_k)
    above = np.full(len(z), np.inf)
    above[passing] = mass_above(z[passing])                 # rule 3b: top-p on the renormalised top-k set
    kept = above < top_p
    near = (np.abs(above - top_p) <= DELTA) & (above > 0) if top_p < 1.0 else np.zeros_like(kept)
    hi = np.nonzero(kept | near)[0]
    g = host_gumbel(host_words(hi, row, step, seed))
    key = z[hi] + g
    in_kept = kept[hi]
    pick = int(hi[np.argmax(np.where(in_kept, key, -np.inf))])        # first maximum = smallest index
    lo_max = np.max(np.where(in_kept & ~near[hi], key, -np.inf))
    eps = EPS_SCALE * (2.0 + float(np.max(np.abs(z[hi]) + np.abs(g))))
    cands = set(int(i) for i in hi[key >= lo_max - eps])
    return pick, cands, passing


def brute_force(x_row, temperature, top_k, top_p, seed, step, row):
    """The rule written out token by token (x_row already guarded): kept set and the Gumbel-max pick."""
    z = [float(np.float32(np.float32(v) / np.float32(temperature))) for v in x_row]
    V = len(z)
    kth = sorted(z, reverse=True)[top_k - 1] if 0 < top_k < V else -math.inf
    passing = [v >= kth for v in z]
    zmax = max(z)
    e = [math.exp(v - zmax) for v in z]
    s = sum(e[j] for j in range(V) if passing[j])
    kept = [passing[i] and sum(e[j] for j in range(V) if passing[j] and z[j] > z[i]) / s < top_p for i in range(V)]
    best, best_i = -math.inf, None
    for i in range(V):
        if not kept[i]:
            continue
        w = int(philox4x32_10(np.array([[i >> 2, row, step, TAG]], np.uint32), (seed & 0xFFFFFFFF, seed >> 32))[0, i & 3])
        u = ((w >> 8) + 0.5) / 2 ** 24
        k = z[i] - math.log(-math.log(u))
        if k > best:
            best, best_i = k, i
    return best_i, np.array(kept), np.array(passing)


# --------------------------------------------------------------------------------------------------------------------
# host finalize (the "after the last step" rule, N best)
# --------------------------------------------------------------------------------------------------------------------
class Image:
    """One image's beam state on the host: running scores s[K]; finished slots [score, len, seq, src] in slot order."""

    def __init__(self, K, s, hyps, count, done):
        self.K, self.s = K, list(s)
        self.hyps = [list(h) for h in hyps]
        self.count, self.done = count, done

    def offer(self, score, length, src):
        K = self.K
        if len(self.hyps) < K:
            self.hyps.append([score, length, self.count, src])
            self.count += 1
            return
        w = min(range(K), key=lambda j: (self.hyps[j][0], self.hyps[j][2]))
        if score > self.hyps[w][0]:
            self.hyps[w] = [score, length, self.count, src]
            self.count += 1


def norm_den32(n: int, alpha: float) -> np.float32:
    return np.float32(min(max(np.float32(n) ** np.float32(alpha), np.finfo(np.float32).tiny), np.finfo(np.float32).max))


def host_finalize_top(img: Image, steps: int, alpha: float, N: int):
    """[(src, len, score)] of the N best after the offers, best first, by selection as the rule states it: each
    pick is the best remaining entry (score desc, then the one added first). Scores are fp32."""
    tmp = Image(img.K, img.s, [h[:3] + [("hyp", j)] for j, h in enumerate(img.hyps)], img.count, img.done)
    if not img.done:
        den = norm_den32(steps, alpha)
        for k in range(img.K):
            tmp.offer(np.float32(np.float32(img.s[k]) / den), steps + 1, ("beam", k))
    left, out = list(range(len(tmp.hyps))), []
    for _ in range(N):
        w = min(left, key=lambda j: (-tmp.hyps[j][0], tmp.hyps[j][2]))
        left.remove(w)
        out.append((tmp.hyps[w][3], tmp.hyps[w][1], tmp.hyps[w][0]))
    return out


# --------------------------------------------------------------------------------------------------------------------
# CPU tests
# --------------------------------------------------------------------------------------------------------------------
def test_host_topk_sampler_equals_brute_force_on_tiny_rows():
    rng = np.random.default_rng(5)
    rows = [
        np.array([0.5], np.float32),
        np.array([1.0, 1.0, 1.0, 1.0], np.float32),                     # all tied
        np.array([2.0, 1.0, 1.0, 1.0, 0.0, -1.0], np.float32),          # a tie group straddling k = 2, 3
        np.array([0.0, 3.0, 3.0, -2.0, 1.0, 1.0, 1.0], np.float32),     # ties at k = 1..2 and 3..5
        rng.standard_normal(8).astype(np.float32),
        (np.round(rng.standard_normal(9) * 2) / 2).astype(np.float32),
        np.array([1.0, np.nan, 2.0, -1.0, 0.5], np.float32),            # NaN row: all zeros, every token ties
        np.array([1.0, np.inf, 2.0, -np.inf, 0.5, 100.0], np.float32),  # Inf row: clamped, ties at 100
    ]
    n = 0
    for x in rows:
        x = host_guard(x[None, :])[0]
        V = len(x)
        for top_k in sorted({0, 1, 2, 3, max(V - 1, 0), V, V + 5}):
            for temperature in (0.3, 1.0):
                for top_p in (1e-9, 0.5, 0.9, 1.0):
                    for step in range(3):
                        want, kept, passing = brute_force(x, temperature, top_k, top_p, 0x0123456789ABCDEF, step, 5)
                        got, cands, hpass = host_sample(x, temperature, top_k, top_p, 0x0123456789ABCDEF, step, 5)
                        assert np.array_equal(hpass, passing), (x, top_k)
                        assert got == want and want in cands, (x, top_k, temperature, top_p, step)
                        assert kept[want] and passing[want]
                        n += 1
    assert n > 600
    z = host_z(rows[2], 1.0)
    assert list(topk_pass(z, 2)) == [True, True, True, True, False, False]      # ties with the k-th pass together
    assert list(topk_pass(z, 1)) == [True, False, False, False, False, False]
    assert topk_pass(host_z(host_guard(rows[6][None])[0], 1.0), 1).all()       # NaN row: every token passes
    assert list(topk_pass(host_z(host_guard(rows[7][None])[0], 1.0), 1)) == [False, True, False, False, False, True]


def test_host_finalize_top_equals_a_full_sort():
    rng = np.random.default_rng(7)
    n = 0
    for trial in range(400):
        K = int(rng.integers(1, 9))
        steps = int(rng.integers(1, 9))
        alpha = float(rng.choice([0.0, 1.0, 2.0]))
        nh = int(rng.integers(0, K + 1))
        done = nh == K and bool(rng.integers(0, 2))
        # scores on a coarse grid: ties between finished entries and with the running beams are common
        hs = [float(np.float32(-rng.integers(0, 12) / 4)) for _ in range(nh)]
        seqs = list(rng.permutation(nh + int(rng.integers(0, 3)))[:nh])
        hyps = [[hs[j], int(rng.integers(1, steps + 1)), int(seqs[j])] for j in range(nh)]
        count = (max(seqs) + 1) if nh else 0
        s = [float(np.float32(-rng.integers(0, 12) / 2 * norm_den32(steps, alpha))) for _ in range(K)]
        img = Image(K, s, hyps, count, done)
        for N in range(1, K + 1):
            got = host_finalize_top(img, steps, alpha, N)
            # the full sort of the set after the offers
            tmp = Image(K, s, [h + [("hyp", j)] for j, h in enumerate(hyps)], count, done)
            if not done:
                den = norm_den32(steps, alpha)
                for k in range(K):
                    tmp.offer(np.float32(np.float32(s[k]) / den), steps + 1, ("beam", k))
            assert len(tmp.hyps) == K                                   # N <= K entries always exist
            full = sorted(tmp.hyps, key=lambda h: (-h[0], h[2]))
            assert got == [(h[3], h[1], h[0]) for h in full[:N]]
            assert all(a[2] >= b[2] for a, b in zip(got, got[1:]))
            n += 1
    assert n > 1000


@pytest.fixture(scope="module")
def lib():
    from vlm_bridge_b200 import _lib, build

    h = C.CDLL(build.build())
    _lib._declare(h)
    h.b200b_sample_tokens.restype = C.c_int
    h.b200b_sample_tokens.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_float, C.c_float,
                                      C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
    h.b200b_last_error.restype = C.c_char_p
    return h


def test_sample_tokens_top_k_argument_codes_need_no_gpu(lib):
    """Every call here fails a host check (the dummy pointers are never handed to a kernel)."""
    buf = C.create_string_buffer(64)
    a = C.addressof(buf)
    ok = dict(logits=a, dtype=0, ld=8, rows=4, vocab=8, temperature=1.0, top_k=3, top_p=0.9, seed=a, step=0, ids=a,
              stride=1)

    def call(**kw):
        g = dict(ok, **kw)
        return lib.b200b_sample_tokens_top_k(g["logits"], g["dtype"], g["ld"], g["rows"], g["vocab"], g["temperature"],
                                             g["top_k"], g["top_p"], g["seed"], g["step"], g["ids"], g["stride"], None)

    for k in ("logits", "seed", "ids"):
        assert call(**{k: None}) == ERR_ARG and b"null" in lib.b200b_last_error()
    for k in (-1, -50, -(1 << 62)):
        assert call(top_k=k) == ERR_ARG and b"top_k" in lib.b200b_last_error()
    assert call(dtype=2) == ERR_ARG
    assert call(ld=7) == ERR_ARG
    assert call(temperature=0.0) == ERR_ARG
    assert call(top_p=0.0) == ERR_ARG and call(top_p=1.5) == ERR_ARG
    assert call(rows=0) == ERR_SHAPE
    # any top_k >= 0 is accepted: these fail only at the vocabulary limit, the last host check
    for k in (0, 1, 360449, 1 << 40):
        assert call(top_k=k, vocab=360449, ld=360449) == ERR_SHAPE and b"exceeds" in lib.b200b_last_error()


def test_beam_finalize_top_argument_codes_need_no_gpu(lib):
    from vlm_bridge_b200 import _lib

    buf = C.create_string_buffer(64)
    a = C.addressof(buf)
    st = _lib.BeamState(a, a, a, a, a, a, a, 5)
    ok = dict(batch=2, K=3, N=2, eos=1, alpha=1.0, steps=4, ids=a, ld_ids=5, state=st, out=a, ld_out=5, out_len=a,
              out_score=a)

    def call(**kw):
        g = dict(ok, **kw)
        return lib.b200b_beam_finalize_top(g["batch"], g["K"], g["N"], g["eos"], g["alpha"], g["steps"], g["ids"],
                                           g["ld_ids"], C.byref(g["state"]), g["out"], g["ld_out"], g["out_len"],
                                           g["out_score"], None)

    for k in ("ids", "out", "out_len", "out_score"):
        assert call(**{k: None}) == ERR_ARG and b"null" in lib.b200b_last_error()
    assert call(state=_lib.BeamState(a, a, a, a, None, a, a, 5)) == ERR_ARG
    for K, N in ((3, 0), (3, 4), (1, 2), (8, 9), (3, -1)):
        assert call(K=K, N=N) == ERR_ARG and b"num_return" in lib.b200b_last_error(), (K, N)
    assert call(K=0, N=1) == ERR_ARG and call(K=9, N=1) == ERR_ARG
    # N in [1, K] passes that check; each of these fails a later one
    for N in (1, 3):
        assert call(N=N, batch=0) == ERR_SHAPE
        assert call(N=N, steps=0) == ERR_SHAPE
        assert call(N=N, ld_out=4) == ERR_ARG
        assert call(N=N, alpha=math.nan) == ERR_ARG


def test_decode_num_return_sequences_and_top_k_raise_value_error():
    from vlm_bridge_b200 import BridgeLite, beam_search_decode, greedy_decode

    m = BridgeLite(vision_dim=32, language_dim=64, num_heads_cross=1, num_heads_self=1)
    v = torch.randn(1, 4, 32)
    fns = (lambda t: torch.zeros(t.shape + (64,)), lambda y: y[:, -1, :])
    kw = dict(bos_token_id=2, max_new_tokens=2)
    for k in (-1, 1.5, "3", True, None):
        with pytest.raises(ValueError, match="top_k"):
            greedy_decode(m, v, *fns, do_sample=True, top_k=k, **kw)
    for n in (0, 9, -1, 2.0, True):
        with pytest.raises(ValueError, match="num_return_sequences"):
            greedy_decode(m, v, *fns, do_sample=True, num_return_sequences=n, **kw)
    with pytest.raises(ValueError, match="do_sample"):
        greedy_decode(m, v, *fns, num_return_sequences=2, **kw)
    with pytest.raises(ValueError, match="use_cache"):
        greedy_decode(m, v, *fns, do_sample=True, num_return_sequences=2, use_cache=False, **kw)
    # greedy decode ignores top_k (validated with do_sample=True only), as it ignores temperature / top_p
    with pytest.raises(RuntimeError, match="CUDA"):
        greedy_decode(m, v, *fns, top_k=-1, **kw)
    for n in (0, 3, -1, 1.5):
        with pytest.raises(ValueError, match="num_return_sequences"):
            beam_search_decode(m, v, *fns, num_beams=2, num_return_sequences=n, bos_token_id=2)
    assert m.training                                   # the mode is restored on the error path


# --------------------------------------------------------------------------------------------------------------------
# GPU, op level
# --------------------------------------------------------------------------------------------------------------------
ROWS = (1, 3, 32, 64)
TEMPS = (0.3, 1.0)
TOPPS = (1e-6, 0.9, 1.0)


def _ks(V):
    return sorted({1, 2, 50, V - 1, V} - {0})


def _logits(rows, vocab, seed, top_k, tdt):
    """float32 [rows, V] representable in tdt: Gaussian rows (scale 3), every other row rounded to quarters; in each
    row up to three more tokens are set to the row's top_k-th largest value (duplicates at the k-th rank); with >= 3
    rows, row 1 holds an Inf and row 2 a NaN."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(rows, vocab, generator=g) * 3.0
    x[1::2] = torch.round(x[1::2] * 4.0) / 4.0
    x = x.to(tdt).float()
    if 1 < top_k < vocab:
        kth = torch.sort(x, dim=1, descending=True).values[:, top_k - 1]
        for j in range(min(3, vocab - top_k)):
            idx = torch.randint(0, vocab, (rows,), generator=g)
            x[torch.arange(rows), idx] = kth
    if rows >= 3:
        x[1, vocab // 2] = math.inf
        x[2, (vocab * 2) // 3] = math.nan
    return x


def _run_case(dtype, vocab, rows, temperature, top_k, top_p, case):
    from vlm_bridge_b200 import ops

    pad = 8 if case % 2 == 0 else 13
    tdt = torch.float32 if dtype == "f32" else torch.bfloat16
    x = _logits(rows, vocab, 2000 + case, top_k, tdt)
    buf = torch.full((rows, vocab + pad), math.nan, dtype=tdt, device="cuda")
    buf[:, :vocab] = x.to(tdt).cuda()
    seen = buf[:, :vocab].float().cpu().numpy()                 # the values the kernel reads
    ids_buf = torch.full((3 * rows + 5,), SENT, dtype=torch.int64, device="cuda")
    out = ids_buf[2:2 + 3 * rows:3]
    seed_val = (0x9E3779B97F4A7C15 * (case + 3)) & 0x7FFFFFFFFFFFFFFF
    seed = torch.tensor([seed_val], dtype=torch.int64, device="cuda")
    step = 3 + case
    ops.sample_tokens(buf[:, :vocab], temperature=temperature, top_k=top_k, top_p=top_p, seed=seed, step=step, out=out)
    got = ids_buf.cpu()
    mask = torch.ones_like(got, dtype=torch.bool)
    mask[2:2 + 3 * rows:3] = False
    assert bool((got[mask] == SENT).all()), "a write outside ids_out"
    got = got[2:2 + 3 * rows:3].numpy()
    xg = host_guard(seen)
    exact = 0
    for b in range(rows):
        pick, cands, passing = host_sample(xg[b], temperature, top_k, top_p, seed_val, step, b)
        where = (dtype, vocab, rows, temperature, top_k, top_p, b)
        assert 0 <= int(got[b]) < vocab and passing[int(got[b])], where          # the top-k threshold is exact
        if len(cands) == 1:
            assert int(got[b]) == pick, where
            exact += 1
        else:
            assert int(got[b]) in cands, where
    return exact, rows


def _cases(dtype, vocab):
    grid = [(r, t, k, p) for r in ROWS for t in TEMPS for k in _ks(vocab) for p in TOPPS]
    if vocab <= 32000:
        return grid if vocab <= 1000 else grid[(0 if dtype == "f32" else 1)::2]
    # 256000 / 256001: every (rows, k) pair once per dtype and vocabulary, (T, top_p) cycling (the float64 host
    # reference of a 64 x 256000 case takes seconds)
    off = (0 if dtype == "f32" else 3) + (0 if vocab == 256000 else 1)
    return [(r, TEMPS[(off + j) % 2], k, TOPPS[(off + j) % 3])
            for j, (r, k) in enumerate((r, k) for r in ROWS for k in _ks(vocab))]


@gpu
@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("vocab", [7, 1000, 32000, 256000, 256001])
def test_sample_tokens_top_k_token_for_token(dtype, vocab):
    exact = total = 0
    for case, (rows, t, k, p) in enumerate(_cases(dtype, vocab)):
        e, n = _run_case(dtype, vocab, rows, t, k, p, case)
        exact += e
        total += n
    print(f"sample_tokens top_k {dtype} V={vocab}: {exact} / {total} rows decided exactly")
    assert exact >= 0.95 * total


@gpu
def test_top_k_zero_or_at_least_vocab_equals_the_top_p_entry(lib):
    from vlm_bridge_b200 import ops

    for vocab, rows, dt in ((7, 3, torch.float32), (1000, 32, torch.bfloat16), (32000, 64, torch.float32),
                            (256001, 3, torch.bfloat16), (256000, 32, torch.float32)):
        x = _logits(rows, vocab, vocab, 0, dt).to(dt).cuda()
        seed = torch.tensor([vocab * 7919], dtype=torch.int64, device="cuda")
        for t, p in ((0.3, 0.9), (1.0, 1.0), (1.0, 1e-6)):
            old = torch.full((rows,), SENT, dtype=torch.int64, device="cuda")
            assert lib.b200b_sample_tokens(x.data_ptr(), 1 if dt == torch.bfloat16 else 0, x.stride(0), rows, vocab,
                                           t, p, seed.data_ptr(), 9, old.data_ptr(), 1,
                                           C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
            for k in (0, vocab, vocab + 1, 1 << 40):
                got = ops.sample_tokens(x, temperature=t, top_k=k, top_p=p, seed=seed, step=9)
                assert torch.equal(got, old), (vocab, dt, t, p, k)


def _draws(x_row, temperature, top_k, top_p, rows=4096, steps=16):
    from vlm_bridge_b200 import ops

    x = torch.as_tensor(x_row, dtype=torch.float32).cuda().repeat(rows, 1)
    seed = torch.tensor([4242], dtype=torch.int64, device="cuda")
    out = torch.empty((steps, rows), dtype=torch.int64, device="cuda")
    for t in range(steps):
        ops.sample_tokens(x, temperature=temperature, top_k=top_k, top_p=top_p, seed=seed, step=t, out=out[t])
    return np.bincount(out.flatten().cpu().numpy(), minlength=len(x_row))


@gpu
def test_sample_tokens_top_k_distribution():
    """2^16 draws per case against the softmax restricted to the k largest (chi-square p > 1e-3, nothing outside)."""
    from scipy.stats import chisquare

    x = (np.linspace(2.5, -2.5, 64)).astype(np.float32)
    x[5] = x[4]                                          # a tie at the 5th value: k = 5 keeps six tokens
    x = np.random.default_rng(1).permutation(x)
    n = 4096 * 16
    for top_k in (1, 5, 50):
        counts = _draws(x, 1.0, top_k, 1.0)
        z = host_z(x, 1.0)
        passing = topk_pass(z, top_k)
        assert passing.sum() == {1: 1, 5: 6, 50: 50}[top_k]
        assert counts.sum() == n and counts[~passing].sum() == 0, (top_k, counts)
        if top_k == 1:
            continue
        q = np.where(passing, np.exp(z - z.max()), 0.0)
        q /= q.sum()
        assert chisquare(counts[passing], q[passing] * n).pvalue > 1e-3, (top_k, counts)


@gpu
def test_sample_tokens_top_k_deterministic_and_graph_reads_the_seed():
    from vlm_bridge_b200 import ops

    rows, vocab, t, k, p = 8, 32000, 1.0, 50, 0.9
    x = _logits(rows, vocab, 5, k, torch.float32)
    x[1:3] = x[3:5]                                      # no NaN / Inf rows here
    xd = x.cuda()
    seed = torch.tensor([1], dtype=torch.int64, device="cuda")
    a = ops.sample_tokens(xd, temperature=t, top_k=k, top_p=p, seed=seed, step=4)
    b = ops.sample_tokens(xd, temperature=t, top_k=k, top_p=p, seed=seed, step=4)
    assert torch.equal(a, b)
    out = torch.empty(rows, dtype=torch.int64, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.sample_tokens(xd, temperature=t, top_k=k, top_p=p, seed=seed, step=4, out=out)   # warm-up outside capture
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ops.sample_tokens(xd, temperature=t, top_k=k, top_p=p, seed=seed, step=4, out=out)
    xs = x.numpy()
    seen = []
    for sv in (1, 2, 0x7FFF0000DEADBEEF):
        seed.fill_(sv)
        graph.replay()
        got = out.cpu().numpy()
        seen.append(tuple(got))
        for r in range(rows):
            pick, cands, passing = host_sample(xs[r], t, k, p, sv, 4, r)
            assert passing[int(got[r])]
            assert int(got[r]) == pick if len(cands) == 1 else int(got[r]) in cands
    assert seen[0] == tuple(a.cpu().numpy())
    assert len(set(seen)) == 3


def _beam_states(B, K, V, T, alpha, early, seed):
    """Run T real beam steps on random logits (EOS boosted so that images finish: strongly with early stopping, which
    then marks them done); returns (ids, state, eos)."""
    from vlm_bridge_b200 import ops

    g = torch.Generator().manual_seed(seed)
    eos = 1
    ids = torch.full((B * K, T + 1), 2, dtype=torch.int64, device="cuda")
    nxt = torch.empty_like(ids)
    par = torch.empty(B * K, dtype=torch.int64, device="cuda")
    st = ops.BeamState(B, K, T + 1, "cuda")
    for t in range(T):
        x = torch.randn(B * K, V, generator=g) * 2.0
        x[:, eos] += torch.rand(B * K, generator=g) * 4.0 + (2.0 if early else -1.0)
        x[::3] = torch.round(x[::3] * 2) / 2                    # ties
        ops.beam_step(x.cuda(), ids, nxt, par, st, step=t, eos_token_id=eos, length_penalty=alpha,
                      early_stopping=early)
        ids, nxt = nxt, ids
    return ids, st, eos


def _host_images(st, B, K):
    s = st.beam_scores.cpu().numpy()
    hs, hl, hq = st.hyp_scores.cpu().numpy(), st.hyp_lens.cpu().numpy(), st.hyp_seq.cpu().numpy()
    cnt, done = st.hyp_count.cpu().numpy(), st.done.cpu().numpy()
    imgs = []
    for b in range(B):
        nh = min(max(int(cnt[b]), 0), K)
        hyps = [[np.float32(hs[b * K + j]), int(hl[b * K + j]), int(hq[b * K + j])] for j in range(nh)]
        imgs.append(Image(K, s[b * K:(b + 1) * K], hyps, int(cnt[b]), bool(done[b])))
    return imgs


@gpu
def test_beam_finalize_top_matches_the_host_ordering(lib):
    from vlm_bridge_b200 import ops

    n_done = n_live = 0
    for case, (B, K, V, T, alpha, early) in enumerate(((16, 4, 64, 6, 1.0, True), (16, 4, 64, 6, 0.0, False),
                                                       (8, 8, 300, 9, 2.0, True), (8, 3, 17, 5, 1.0, False),
                                                       (4, 1, 40, 4, 1.0, True))):
        ids, st, eos = _beam_states(B, K, V, T, alpha, early, 30 + case)
        imgs = _host_images(st, B, K)
        hyp_ids = st.hyp_ids.cpu()
        run_ids = ids.cpu()
        n_done += sum(im.done for im in imgs)
        n_live += sum(not im.done for im in imgs)
        # N = 1 through the wrapper and through the N = 1 entry point: the same bits
        one = ops.beam_finalize(ids, st, steps=T, eos_token_id=eos, length_penalty=alpha)
        o_ids = torch.full((B, T + 1), SENT, dtype=torch.int64, device="cuda")
        o_len = torch.full((B,), SENT, dtype=torch.int64, device="cuda")
        o_sc = torch.full((B,), math.nan, dtype=torch.float32, device="cuda")
        assert lib.b200b_beam_finalize(B, K, eos, alpha, T, ids.data_ptr(), ids.stride(0), C.byref(st.struct),
                                       o_ids.data_ptr(), o_ids.stride(0), o_len.data_ptr(), o_sc.data_ptr(),
                                       C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
        for a, b in zip(one, (o_ids, o_len, o_sc)):
            assert torch.equal(a, b)
        for N in sorted({1, K}):
            g_ids, g_len, g_sc = (t.cpu() for t in ops.beam_finalize(ids, st, steps=T, eos_token_id=eos,
                                                                     length_penalty=alpha, num_return_sequences=N))
            assert g_ids.shape == (B * N, T + 1) and g_len.shape == g_sc.shape == (B * N,)
            for b in range(B):
                want = host_finalize_top(imgs[b], T, alpha, N)
                for j, (src, ln, sc) in enumerate(want):
                    r = b * N + j
                    assert int(g_len[r]) == ln and np.float32(g_sc[r]) == np.float32(sc), (case, N, b, j)
                    row = hyp_ids[b * K + src[1]] if src[0] == "hyp" else run_ids[b * K + src[1]]
                    assert torch.equal(g_ids[r, :ln], row[:ln]), (case, N, b, j)
                    assert bool((g_ids[r, ln:] == eos).all())
            assert torch.equal(g_ids[::N], one[0].cpu()) and torch.equal(g_len[::N], one[1].cpu())
            assert torch.equal(g_sc[::N], one[2].cpu())
    assert n_done >= 4 and n_live >= 4, (n_done, n_live)


# --------------------------------------------------------------------------------------------------------------------
# GPU, end to end (the stand-in language model of test_sampling_gpu.py, at a reduced size)
# --------------------------------------------------------------------------------------------------------------------
E2E_B, E2E_NV, E2E_STEPS, E2E_V = 3, 33, 6, 512


def _e2e_setup(B=E2E_B):
    from oracle import bridge_oracle as O
    from vlm_bridge_b200 import BridgeLite

    sd = O.init_state_dict(1)
    g = torch.Generator().manual_seed(20)
    vision = torch.randn(B, E2E_NV, 1024, generator=g).cuda()
    embed = torch.randn(E2E_V, 2304, generator=g).cuda()
    head = (torch.randn(E2E_V, 2304, generator=g) / 48.0).cuda()
    m = BridgeLite(dropout=0.0)
    m.load_state_dict(sd, strict=True)
    return m.cuda().eval(), vision, embed, head, (lambda t: embed[t]), (lambda y: y[:, -1, :] @ head.t())


@gpu
def test_sampled_num_return_sequences_equals_the_repeated_batch_fp32():
    """N samples per image over the shared cache equal a sampled decode over the images repeated N times, token for
    token (fp32: the bridge output is bit-equal across the two cache layouts), eagerly and with step graphs."""
    from vlm_bridge_b200 import VisionKVCache, greedy_decode
    from vlm_bridge_b200.decode import DecodeStepGraphs

    m, vision, _, _, ef, lf = _e2e_setup()
    kw = dict(bos_token_id=2, eos_token_id=1, max_new_tokens=E2E_STEPS, do_sample=True, precision="fp32")
    gen = torch.Generator(device="cuda")
    for N, t, k, p in ((5, 1.3, 50, 0.9), (2, 0.8, 0, 1.0), (8, 1.0, 3, 0.95)):
        rep = vision.repeat_interleave(N, 0)
        gen.manual_seed(N)
        want, wl = greedy_decode(m, rep, ef, lf, temperature=t, top_k=k, top_p=p, generator=gen, **kw)
        gen.manual_seed(N)
        got, gl = greedy_decode(m, vision, ef, lf, temperature=t, top_k=k, top_p=p, num_return_sequences=N,
                                generator=gen, **kw)
        assert got.shape == (E2E_B * N, E2E_STEPS + 1)
        assert torch.equal(got, want) and torch.equal(gl, wl), (N, t, k, p)
        cache = VisionKVCache(m, vision, precision="fp32", beams=N)
        graphs = DecodeStepGraphs(m, cache)
        for _ in range(2):                                        # capture, then replay
            gen.manual_seed(N)
            gg, gl2 = greedy_decode(m, vision, ef, lf, temperature=t, top_k=k, top_p=p, num_return_sequences=N,
                                    generator=gen, kv_cache=cache, step_graphs=graphs, **kw)
            assert torch.equal(gg, want) and torch.equal(gl2, wl), (N, "graphs")
    # the N samples of an image differ (a temperature of 1.3 over 512 tokens)
    assert len({tuple(r) for r in got.view(E2E_B, 8, -1)[0].tolist()}) > 1


@gpu
def test_sampled_num_return_sequences_has_no_host_sync():
    from vlm_bridge_b200 import VisionKVCache, greedy_decode
    from vlm_bridge_b200.decode import DecodeStepGraphs

    m, vision, _, _, ef, lf = _e2e_setup()
    N = 4
    cache = VisionKVCache(m, vision, beams=N)
    graphs = DecodeStepGraphs(m, cache)
    gen = torch.Generator(device="cuda").manual_seed(3)
    kw = dict(bos_token_id=2, eos_token_id=1, max_new_tokens=E2E_STEPS, kv_cache=cache, do_sample=True,
              temperature=0.9, top_k=50, top_p=0.9, num_return_sequences=N, generator=gen)
    greedy_decode(m, vision, ef, lf, **kw)                          # lazy initialisation
    greedy_decode(m, vision, ef, lf, step_graphs=graphs, **kw)      # graph capture
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        eager, _ = greedy_decode(m, vision, ef, lf, **kw)
        replay, _ = greedy_decode(m, vision, ef, lf, step_graphs=graphs, use_graphs=True, **kw)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert eager.shape == replay.shape == (E2E_B * N, E2E_STEPS + 1)
    with pytest.raises(ValueError, match="beams=4, this decode runs 2"):     # a cache built for other beams
        greedy_decode(m, vision, ef, lf, **dict(kw, num_return_sequences=2))


@gpu
def test_top_k_1_sampling_is_greedy():
    """top_k = 1 keeps only the maximum, so a sampled decode at any temperature is the greedy one on rows whose
    maximum is unique (a tied maximum keeps every tied token; the seeded logits of this model have none)."""
    from vlm_bridge_b200 import greedy_decode

    m, vision, _, _, ef, lf = _e2e_setup()
    kw = dict(bos_token_id=2, eos_token_id=1, max_new_tokens=E2E_STEPS)
    for precision in ("bf16", "fp32"):
        ids_g, len_g = greedy_decode(m, vision, ef, lf, precision=precision, **kw)
        for N in (1, 3):
            ids_s, len_s = greedy_decode(m, vision, ef, lf, precision=precision, do_sample=True, temperature=2.0,
                                         top_k=1, num_return_sequences=N, **kw)
            assert torch.equal(ids_s, ids_g.repeat_interleave(N, 0)), (precision, N)
            assert torch.equal(len_s, len_g.repeat_interleave(N, 0))


@gpu
def test_beam_search_num_return_sequences():
    """Row b*N equals the N = 1 result, scores are non-increasing within an image, and every returned hypothesis'
    score is its teacher-forced log-probability (EOS included) over n ** alpha, within the C4 beam test's bound."""
    from vlm_bridge_b200 import VisionKVCache, beam_search_decode

    B, K, T = 4, 4, 8
    m, vision, embed, head, ef, lf = _e2e_setup(B)
    kw = dict(num_beams=K, bos_token_id=2, eos_token_id=1, max_new_tokens=T, length_penalty=1.0, precision="fp32")
    one = beam_search_decode(m, vision, ef, lf, **kw)
    for N in (1, 2, K):
        ids, lengths, scores = beam_search_decode(m, vision, ef, lf, num_return_sequences=N, **kw)
        assert ids.shape == (B * N, T + 1) and lengths.shape == scores.shape == (B * N,)
        for a, b in zip((ids[::N], lengths[::N], scores[::N]), one):
            assert torch.equal(a, b), N
        sc = scores.view(B, N)
        assert bool((sc[:, 1:] <= sc[:, :-1]).all()), sc
        if N < K:
            continue
        n = torch.where(lengths <= T, lengths, lengths - 1)
        total = torch.zeros(B * N, dtype=torch.float64, device="cuda")
        c32 = VisionKVCache(m, vision.repeat_interleave(N, 0), max_positions=0, precision="fp32")
        with torch.no_grad():
            for j in range(T):
                y = m(None, embed[ids[:, :j + 1]], kv_cache=c32)
                logp = torch.log_softmax(y[:, -1, :] @ head.t(), dim=-1)
                lp = logp.gather(1, ids[:, j + 1:j + 2])[:, 0].double()
                total += torch.where(j < n, lp, torch.zeros_like(lp))
        want = total / n.double()
        err = (scores.double() - want).abs()
        print(f"beam num_return_sequences={N}: largest |score - teacher-forced score| = {float(err.max()):.2e}")
        assert bool((err <= 1e-3 * want.abs().clamp(min=1.0)).all()), (scores, want)
