"""Temperature / top-p sampling (csrc/sampling.cu, ops.sample_tokens, greedy_decode(do_sample=True)).

The rule (include/b200_bridge.h, b200b_sample_tokens) fixes every random number: token i of row b at step t uses
the Philox4x32-10 word i % 4 of counter (i / 4, b, t, 0x5a3b1e00) under the 64-bit seed, and the draw is the
Gumbel-max argmax over the nucleus. So the kernel is checked token for token against a float64 host sampler fed
with the same Philox words (the numpy Philox of test_gemm_ops_gpu, pinned there to the Random123 known answers).
The host divides by the temperature in fp32, as the rule says, so host and kernel order the tokens by the same z
values; everything after that is float64 on the host.

A kernel id may differ from the host's only where fp32 rounding can decide, and then it must be a candidate:
  * EPS (Gumbel keys): the kernel's key z + g differs from the host's by the log errors and one rounding. logf /
    log1pf are within 1 ulp (2^-23 relative) of -ln u and of ln(-ln u), and z + g is rounded once (2^-24 |z + g|):
    |error| <= 2^-22 (1 + |z| + |g|). EPS = 2^-20 (2 + max |z| + |g|) is four times that.
  * DELTA (nucleus edge): the masses are sums of ex2.approx(z - zmax) (relative error ~2^-22, plus |z - zmax|
    2^-23 from rounding the argument: <= 5e-6 for the terms above 2^-40) in 2^-40 fixed point (truncation
    <= V 2^-40 <= 2.4e-7 of a sum that is >= 1). A mass above and the total are each off by < 6e-6, their ratio
    by < 1.2e-5: DELTA = 1e-4. A token whose mass above lies within DELTA of top_p may go either way (the
    maximum, whose mass above is exactly 0, never does).
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import pytest
import torch

from test_gemm_ops_gpu import philox4x32_10

gpu = pytest.mark.gpu
TAG = 0x5A3B1E00
EPS_SCALE = 2.0 ** -20
DELTA = 1e-4
ERR_SHAPE, ERR_ARG = -1, -3
SENT = -7777


# --------------------------------------------------------------------------------------------------------------------
# float64 host sampler
# --------------------------------------------------------------------------------------------------------------------
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


def host_sample(x_row: np.ndarray, temperature: float, top_p: float, seed: int, step: int, row: int):
    """(host pick, candidate ids the kernel may return) for one guarded float32 row."""
    z = host_z(x_row, temperature)
    above = mass_above(z)
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
    return pick, cands


def brute_force(x_row, temperature, top_p, seed, step, row):
    """The rule written out token by token: kept set and the Gumbel-max pick."""
    z = [float(np.float32(np.float32(v) / np.float32(temperature))) for v in x_row]
    zmax = max(z)
    e = [math.exp(v - zmax) for v in z]
    s = sum(e)
    kept = [sum(e[j] for j in range(len(z)) if z[j] > z[i]) / s < top_p for i in range(len(z))]
    best, best_i = -math.inf, None
    for i in range(len(z)):
        if not kept[i]:
            continue
        w = int(philox4x32_10(np.array([[i >> 2, row, step, TAG]], np.uint32),
                              (seed & 0xFFFFFFFF, seed >> 32))[0, i & 3])
        u = ((w >> 8) + 0.5) / 2 ** 24
        k = z[i] - math.log(-math.log(u))
        if k > best:
            best, best_i = k, i
    return best_i, np.array(kept)


# --------------------------------------------------------------------------------------------------------------------
# CPU tests
# --------------------------------------------------------------------------------------------------------------------
def test_host_sampler_equals_brute_force_on_tiny_rows():
    rng = np.random.default_rng(3)
    rows = [
        np.array([0.5], np.float32),
        np.array([1.0, 1.0, 1.0, 1.0], np.float32),                     # all tied
        np.array([2.0, 1.0, 1.0, 0.0, -1.0], np.float32),               # a tie group straddling the threshold
        np.array([0.0, 3.0, 3.0, -2.0, 1.0, 1.0, 1.0], np.float32),
        rng.standard_normal(8).astype(np.float32),
        (np.round(rng.standard_normal(8) * 2) / 2).astype(np.float32),
    ]
    n = 0
    for x in rows:
        for temperature in (0.3, 1.0, 1.7):
            for top_p in (1e-9, 0.3, 0.5, 0.75, 0.9, 1.0):
                for step in range(6):
                    want, kept = brute_force(x, temperature, top_p, 0x0123456789ABCDEF, step, 5)
                    got, cands = host_sample(x, temperature, top_p, 0x0123456789ABCDEF, step, 5)
                    z = host_z(x, temperature)
                    assert np.array_equal(mass_above(z) < top_p, kept)
                    assert got == want and want in cands
                    n += 1
    assert n == 6 * 3 * 6 * 6
    # the tie group {1, 2} of row 2 (mass above = p(2.0) ~ 0.53) is kept or dropped together
    z = host_z(rows[2], 1.0)
    assert list(mass_above(z) < 0.6) == [True, True, True, False, False]
    assert list(mass_above(z) < 0.5) == [True, False, False, False, False]
    # top_p -> 0 keeps exactly the maximum (all of a tied maximum), top_p = 1 keeps everything
    assert list(mass_above(host_z(rows[3], 1.0)) < 1e-12) == [False, True, True, False, False, False, False]
    assert bool((mass_above(host_z(rows[4], 1.0)) < 1.0).all())


def test_host_sampler_draws_the_renormalised_nucleus():
    """Gumbel-max over the nucleus is an exact draw from it: 40000 host draws against the renormalised nucleus."""
    from scipy.stats import chisquare

    x = np.array([1.2, 0.9, 0.9, 0.2, -0.4, -1.0], np.float32)
    z = host_z(x, 0.8)
    kept = mass_above(z) < 0.8
    q = np.where(kept, np.exp(z - z.max()), 0.0)
    q /= q.sum()
    n = 40000
    idx = np.arange(len(x))
    counts = np.zeros(len(x))
    for step in range(n // 200):
        for row in range(200):
            g = host_gumbel(host_words(idx, row, step, 99))
            counts[int(np.argmax(np.where(kept, z + g, -np.inf)))] += 1
    assert counts[~kept].sum() == 0
    assert chisquare(counts[kept], q[kept] * n).pvalue > 1e-3


@pytest.fixture(scope="module")
def lib():
    from vlm_bridge_b200 import build

    h = C.CDLL(build.build())
    h.b200b_sample_tokens.restype = C.c_int
    h.b200b_sample_tokens.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_float, C.c_float,
                                      C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
    h.b200b_last_error.restype = C.c_char_p
    return h


def test_sample_tokens_argument_codes_need_no_gpu(lib):
    """Every bad argument is rejected on the host before any CUDA call (these pointers are never dereferenced)."""
    buf = C.create_string_buffer(64)
    a = C.addressof(buf)
    ok = dict(logits=a, dtype=0, ld=8, rows=4, vocab=8, temperature=1.0, top_p=0.9, seed=a, step=0, ids=a, stride=1)

    def call(**kw):
        args = dict(ok, **kw)
        return lib.b200b_sample_tokens(args["logits"], args["dtype"], args["ld"], args["rows"], args["vocab"],
                                       args["temperature"], args["top_p"], args["seed"], args["step"], args["ids"],
                                       args["stride"], None)

    assert call(logits=None) == ERR_ARG and b"null" in lib.b200b_last_error()
    assert call(seed=None) == ERR_ARG
    assert call(ids=None) == ERR_ARG
    assert call(dtype=2) == ERR_ARG and b"dtype" in lib.b200b_last_error()
    assert call(dtype=-1) == ERR_ARG
    assert call(ld=7) == ERR_ARG
    for t in (0.0, -1.0, math.inf, math.nan):
        assert call(temperature=t) == ERR_ARG
    for p in (0.0, -0.1, 1.0001, math.inf, math.nan):
        assert call(top_p=p) == ERR_ARG
    assert call(rows=0) == ERR_SHAPE
    assert call(vocab=0, ld=8) == ERR_SHAPE
    # the documented vocabulary limits: 8 * (180224 / e) tokens
    assert call(vocab=360449, ld=360449) == ERR_SHAPE
    assert call(dtype=1, vocab=720897, ld=720897) == ERR_SHAPE
    assert b"exceeds" in lib.b200b_last_error()


def test_greedy_decode_sampling_arguments_raise_value_error():
    from vlm_bridge_b200 import BridgeLite, greedy_decode

    m = BridgeLite(vision_dim=32, language_dim=64, num_heads_cross=1, num_heads_self=1)
    v = torch.randn(1, 4, 32)
    kw = dict(bos_token_id=2, max_new_tokens=2, do_sample=True)
    fns = (lambda t: torch.zeros(t.shape + (64,)), lambda y: y[:, -1, :])
    for t in (0.0, -1.0, math.inf, math.nan):
        with pytest.raises(ValueError, match="temperature"):
            greedy_decode(m, v, *fns, temperature=t, **kw)
    for p in (0.0, 1.5, math.nan):
        with pytest.raises(ValueError, match="top_p"):
            greedy_decode(m, v, *fns, top_p=p, **kw)
    with pytest.raises(ValueError, match="CUDA"):
        greedy_decode(m, v, *fns, **kw)
    assert m.training                                   # the mode is restored on the error path


# --------------------------------------------------------------------------------------------------------------------
# GPU tests
# --------------------------------------------------------------------------------------------------------------------
ROWS = (1, 3, 32, 64)
TEMPS = (0.3, 1.0, 1.7)
TOPPS = (1e-6, 0.5, 0.9, 1.0)


def _logits(rows, vocab, seed):
    """float32 [rows, vocab]: Gaussian rows (scale 3), every other row rounded to quarters (ties at the threshold);
    with >= 3 rows, row 1 holds an Inf and row 2 a NaN."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(rows, vocab, generator=g) * 3.0
    x[1::2] = torch.round(x[1::2] * 4.0) / 4.0
    if rows >= 3:
        x[1, vocab // 2] = math.inf
        x[2, (vocab * 2) // 3] = math.nan
    return x


def _run_case(dtype, vocab, rows, temperature, top_p, case):
    from vlm_bridge_b200 import ops

    pad = 8 if case % 2 == 0 else 13
    x = _logits(rows, vocab, 1000 + case)
    tdt = torch.float32 if dtype == "f32" else torch.bfloat16
    buf = torch.full((rows, vocab + pad), math.nan, dtype=tdt, device="cuda")
    buf[:, :vocab] = x.to(tdt).cuda()
    seen = buf[:, :vocab].float().cpu().numpy()                 # the values the kernel reads
    ids_buf = torch.full((3 * rows + 5,), SENT, dtype=torch.int64, device="cuda")
    out = ids_buf[2:2 + 3 * rows:3]
    seed_val = (0x9E3779B97F4A7C15 * (case + 1)) & 0x7FFFFFFFFFFFFFFF
    seed = torch.tensor([seed_val], dtype=torch.int64, device="cuda")
    step = 5 + case
    ops.sample_tokens(buf[:, :vocab], temperature=temperature, top_p=top_p, seed=seed, step=step, out=out)
    got = ids_buf.cpu()
    mask = torch.ones_like(got, dtype=torch.bool)
    mask[2:2 + 3 * rows:3] = False
    assert bool((got[mask] == SENT).all()), "a write outside ids_out"
    got = got[2:2 + 3 * rows:3].numpy()
    xg = host_guard(seen)
    exact = 0
    for b in range(rows):
        pick, cands = host_sample(xg[b], temperature, top_p, seed_val, step, b)
        if len(cands) == 1:
            assert int(got[b]) == pick, (dtype, vocab, rows, temperature, top_p, b)
            exact += 1
        else:
            assert int(got[b]) in cands, (dtype, vocab, rows, temperature, top_p, b, sorted(cands)[:8])
    return exact, rows


def _cases(dtype, vocab):
    if vocab <= 32000:
        return [(r, t, p) for r in ROWS for t in TEMPS for p in TOPPS]
    # 256000 / 256001: every row count once per dtype, (T, top_p) cycling so that every pair of the grid appears
    # across the two vocabularies and dtypes (the float64 host reference of a 64 x 256000 case takes seconds)
    k0 = (0 if dtype == "f32" else 8) + (0 if vocab == 256000 else 4)
    return [(r, TEMPS[(k0 + j) % 3], TOPPS[(k0 + j) % 4]) for j, r in enumerate(ROWS)]


@gpu
@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("vocab", [1, 7, 1000, 32000, 256000, 256001])
def test_sample_tokens_token_for_token(dtype, vocab):
    exact = total = 0
    for case, (rows, t, p) in enumerate(_cases(dtype, vocab)):
        e, n = _run_case(dtype, vocab, rows, t, p, case)
        exact += e
        total += n
    print(f"sample_tokens {dtype} V={vocab}: {exact} / {total} rows decided exactly")
    assert exact >= 0.99 * total


def _draws(x_row, temperature, top_p, rows=4096, steps=16, dtype=torch.float32):
    from vlm_bridge_b200 import ops

    x = torch.as_tensor(x_row, dtype=torch.float32).to(dtype).cuda().repeat(rows, 1)
    seed = torch.tensor([12345], dtype=torch.int64, device="cuda")
    out = torch.empty((steps, rows), dtype=torch.int64, device="cuda")
    for t in range(steps):
        ops.sample_tokens(x, temperature=temperature, top_p=top_p, seed=seed, step=t, out=out[t])
    return np.bincount(out.flatten().cpu().numpy(), minlength=len(x_row))


@gpu
def test_sample_tokens_distribution():
    """2^16 draws per case against the renormalised nucleus (chi-square p > 1e-3, nothing outside the nucleus)."""
    from scipy.stats import chisquare

    x = np.array([2.0, 1.5, 1.5, 1.0, 0.5, 0.0, -0.5, -1.0, -2.0, -3.0, -4.0, -5.0], np.float32)
    n = 4096 * 16
    for temperature, top_p, dt in ((0.8, 0.7, torch.float32), (1.0, 1.0, torch.float32), (1.7, 0.9, torch.bfloat16),
                                   (0.5, 0.95, torch.float32)):
        counts = _draws(x, temperature, top_p, dtype=dt)
        z = host_z(x, temperature)
        kept = mass_above(z) < top_p
        q = np.where(kept, np.exp(z - z.max()), 0.0)
        q /= q.sum()
        assert counts.sum() == n and counts[~kept].sum() == 0, (temperature, top_p, counts)
        assert chisquare(counts[kept], q[kept] * n).pvalue > 1e-3, (temperature, top_p, counts)
    # a NaN row samples uniformly
    xn = x.copy()
    xn[4] = np.nan
    counts = _draws(xn, 1.0, 0.5)
    assert chisquare(counts, np.full(len(x), n / len(x))).pvalue > 1e-3, counts
    # an Inf row follows the clamp rule: +inf -> 100, -inf -> -100
    xi = x.copy()
    xi[3], xi[7] = np.inf, -np.inf
    counts = _draws(xi, 30.0, 1.0)
    z = host_z(np.clip(xi, -100, 100), 30.0)
    q = np.exp(z - z.max())
    q /= q.sum()
    assert chisquare(counts, q * n).pvalue > 1e-3, counts


@gpu
@pytest.mark.parametrize("vocab", [32000, 256000])
def test_sample_tokens_limits(vocab):
    from vlm_bridge_b200 import ops

    g = torch.Generator().manual_seed(vocab)
    rows = 16
    x = torch.randn(rows, vocab, generator=g) * 2.0
    top = torch.randint(0, vocab, (rows,), generator=g)
    x[torch.arange(rows), top] = x.max(dim=1).values + 1.0       # a unique maximum, 1.0 above the rest
    seed = torch.tensor([77], dtype=torch.int64, device="cuda")
    for dt in (torch.float32, torch.bfloat16):
        xd = x.to(dt).cuda()
        want = torch.argmax(xd.float(), dim=1).cpu()
        assert torch.equal(want, top)
        for t, p in ((1.0, 1e-6), (1.7, 1e-6), (1e-4, 1.0), (1e-4, 0.9)):
            for step in range(3):
                got = ops.sample_tokens(xd, temperature=t, top_p=p, seed=seed, step=step).cpu()
                assert torch.equal(got, want), (dt, t, p)
    # -inf everywhere except one index
    xm = torch.full((rows, vocab), -math.inf)
    xm[torch.arange(rows), top] = torch.randn(rows, generator=g)
    for t, p in ((0.3, 0.5), (1.0, 1.0), (1.7, 0.9)):
        got = ops.sample_tokens(xm.cuda(), temperature=t, top_p=p, seed=seed, step=1).cpu()
        assert torch.equal(got, top)


@gpu
def test_sample_tokens_deterministic_and_graph_reads_the_seed():
    from vlm_bridge_b200 import ops

    rows, vocab, t, p = 8, 32000, 1.0, 0.9
    x = _logits(rows, vocab, 5)
    x[1:3] = x[3:5]                                      # no NaN / Inf rows here
    xd = x.cuda()
    seed = torch.tensor([1], dtype=torch.int64, device="cuda")
    a = ops.sample_tokens(xd, temperature=t, top_p=p, seed=seed, step=4)
    b = ops.sample_tokens(xd, temperature=t, top_p=p, seed=seed, step=4)
    assert torch.equal(a, b)
    out = torch.empty(rows, dtype=torch.int64, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.sample_tokens(xd, temperature=t, top_p=p, seed=seed, step=4, out=out)     # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ops.sample_tokens(xd, temperature=t, top_p=p, seed=seed, step=4, out=out)
    xs = x.numpy()
    seen = []
    for sv in (1, 2, 0x7FFF0000DEADBEEF):
        seed.fill_(sv)
        graph.replay()
        got = out.cpu().numpy()
        seen.append(tuple(got))
        for r in range(rows):
            pick, cands = host_sample(xs[r], t, p, sv, 4, r)
            assert int(got[r]) == pick if len(cands) == 1 else int(got[r]) in cands
    assert seen[0] == tuple(a.cpu().numpy())
    assert len(set(seen)) == 3


# end to end over the stand-in language model of test_decode_c4_gpu.py, at a reduced size
E2E_B, E2E_NV, E2E_STEPS, E2E_V = 4, 33, 6, 512


def _e2e_setup():
    from oracle import bridge_oracle as O
    from vlm_bridge_b200 import BridgeLite

    sd = O.init_state_dict(1)
    g = torch.Generator().manual_seed(20)
    vision = torch.randn(E2E_B, E2E_NV, 1024, generator=g).cuda()
    embed = torch.randn(E2E_V, 2304, generator=g).cuda()
    head = (torch.randn(E2E_V, 2304, generator=g) / 48.0).cuda()
    m = BridgeLite(dropout=0.0)
    m.load_state_dict(sd, strict=True)
    return m.cuda().eval(), vision, (lambda t: embed[t]), (lambda y: y[:, -1, :] @ head.t())


@gpu
def test_greedy_decode_do_sample():
    from vlm_bridge_b200 import greedy_decode

    m, vision, ef, lf = _e2e_setup()
    kw = dict(bos_token_id=2, eos_token_id=1, max_new_tokens=E2E_STEPS)
    for precision in ("bf16", "fp32"):
        ids_g, len_g = greedy_decode(m, vision, ef, lf, precision=precision, **kw)
        ids_s, len_s = greedy_decode(m, vision, ef, lf, precision=precision, do_sample=True, top_p=1e-6, **kw)
        assert torch.equal(ids_g, ids_s) and torch.equal(len_g, len_s), precision
    gen = torch.Generator(device="cuda").manual_seed(7)
    a, la = greedy_decode(m, vision, ef, lf, do_sample=True, temperature=1.5, top_p=0.95, generator=gen, **kw)
    gen.manual_seed(7)
    b, lb = greedy_decode(m, vision, ef, lf, do_sample=True, temperature=1.5, top_p=0.95, generator=gen, **kw)
    c, _ = greedy_decode(m, vision, ef, lf, do_sample=True, temperature=1.5, top_p=0.95, generator=gen, **kw)
    assert torch.equal(a, b) and torch.equal(la, lb)
    assert not torch.equal(a, c)
    # lengths follow the first EOS, as in the greedy path
    for r in range(E2E_B):
        row = a[r, 1:].tolist()
        assert int(la[r]) == ((row.index(1) + 1) if 1 in row else E2E_STEPS + 1)
    with pytest.raises(ValueError, match="generator"):
        greedy_decode(m, vision, ef, lf, do_sample=True, generator=torch.Generator(), **kw)


@gpu
def test_greedy_decode_do_sample_has_no_host_sync():
    from vlm_bridge_b200 import VisionKVCache, greedy_decode
    from vlm_bridge_b200.decode import DecodeStepGraphs

    m, vision, ef, lf = _e2e_setup()
    cache = VisionKVCache(m, vision)
    graphs = DecodeStepGraphs(m, cache)
    gen = torch.Generator(device="cuda").manual_seed(3)
    kw = dict(bos_token_id=2, eos_token_id=1, max_new_tokens=E2E_STEPS, kv_cache=cache, do_sample=True,
              temperature=0.9, top_p=0.9, generator=gen)
    greedy_decode(m, vision, ef, lf, **kw)                          # lazy initialisation
    greedy_decode(m, vision, ef, lf, step_graphs=graphs, **kw)      # graph capture
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        eager, _ = greedy_decode(m, vision, ef, lf, **kw)
        replay, _ = greedy_decode(m, vision, ef, lf, step_graphs=graphs, use_graphs=True, **kw)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert eager.shape == replay.shape == (E2E_B, E2E_STEPS + 1)
