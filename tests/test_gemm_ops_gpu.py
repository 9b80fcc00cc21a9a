"""Op-level parity of the tcgen05 GEMM (csrc/gemm_sm100.cu) and of the dropout masks it shares with the cast kernels.

Two kinds of input:
  * exact by construction -- operands are integers in [-4, 4], bias / residual / beta * out multiples of 1/8 and
    |acc| < 2^20, so every partial sum is exact in fp32 in any order and each output must equal its fp64 reference
    BIT FOR BIT. No tolerance hides a wrong tail row / column, a dropped k block, a pipeline-phase slip or a write to
    the wrong row pitch.
  * realistic -- Gaussian operands (activations sigma 0.5, weights 0.02) at bridge sizes, held to an elementwise
    bound: accumulator |acc - ref| <= 4 sqrt(K) 2^-24 (|A| |B|^T)_ij, plus one bf16 rounding (2^-8 |ref|) for bf16
    outputs. GELU / dGELU outputs are held to one bf16 ulp of fp64 gelu / gelu' of the kernel's own bf16 operand plus
    an absolute floor of 1e-6 max|ref|: gelu_erf uses the Abramowitz-Stegun erfc (common.cuh), whose relative error
    reaches 0.4 bf16 ulp at x = -5 and 2.6 ulp at x = -8, where |gelu| < 1e-14 -- the floor covers that tail, which
    is far below anything the bf16 result of a Linear can resolve.

Every written output sits inside a larger buffer filled with a sentinel (a guard region before the base pointer,
columns right of n inside the pitch, rows below m), and every sentinel byte must survive: weight gradients are written
straight into the flat gradient arena next to other parameters' gradients.

The dropout masks are regenerated on the host by a numpy Philox4x32-10 that is pinned to the Random123 known-answer
vectors (a CPU test), and compared bit for bit with what the GEMM epilogues and the cast kernels apply.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import math

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu

EPI_BF16_BIAS, EPI_BF16_BIAS_GELU, EPI_F32_BIAS_RESID, EPI_BF16_DGELU, EPI_F32 = 0, 1, 2, 3, 4
EPI_NAMES = {0: "bias", 1: "gelu", 2: "resid", 3: "dgelu", 4: "f32"}
SEED_INDIRECT = 0x80000000
ERR_SHAPE, ERR_ALIGN, ERR_ARG = -1, -2, -3

# --------------------------------------------------------------------------------------------------------------------
# host Philox4x32-10 and the dropout mask rule of the library (common.cuh philox4x32_10 / dropout_keep, launch.h
# make_dropout_cfg)
# --------------------------------------------------------------------------------------------------------------------
_MASK32 = np.uint64(0xFFFFFFFF)


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


def dropout_threshold_scale(p: float) -> tuple[int, float]:
    """thr = round(p * 65536) and scale = 1 / (1 - p), both evaluated in fp32 as the library does."""
    p32 = np.float32(p)
    thr = int(np.float32(p32 * np.float32(65536.0)) + np.float32(0.5))
    thr = min(max(thr, 1), 65535)
    return thr, float(np.float32(1.0) / (np.float32(1.0) - p32))


def dropout_keep(numel: int, p: float, seed: int, stream: int) -> np.ndarray:
    """keep[i] for the elements 0..numel-1 of dropout stream `stream`: element i uses 16-bit lane i % 8 of Philox of
    counter (i // 8 low, i // 8 high, stream, 0x0b200b00) and key (seed low, seed high); kept iff lane >= thr."""
    thr, _ = dropout_threshold_scale(p)
    groups = (numel + 7) // 8
    g = np.arange(groups, dtype=np.uint64)
    ctr = np.empty((groups, 4), np.uint32)
    ctr[:, 0] = (g & _MASK32).astype(np.uint32)
    ctr[:, 1] = (g >> np.uint64(32)).astype(np.uint32)
    ctr[:, 2] = stream
    ctr[:, 3] = 0x0B200B00
    words = philox4x32_10(ctr, (seed & 0xFFFFFFFF, seed >> 32))
    lanes = np.stack([words & 0xFFFF, words >> 16], -1).reshape(groups, 8)   # element e: word e // 2, high half if odd
    return lanes.reshape(-1)[:numel] >= thr


def test_philox_known_answers():
    """The host Philox reproduces the Random123 known-answer vectors (kat_vectors, philox4x32_10)."""
    cases = [
        ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
        ((0xFFFFFFFF,) * 4, (0xFFFFFFFF, 0xFFFFFFFF), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
        ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
         (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
    ]
    for ctr, key, want in cases:
        got = philox4x32_10(np.array([ctr], dtype=np.uint32), key)[0]
        assert [int(v) for v in got] == list(want)
    # batched evaluation is element-wise
    ctrs = np.array([c for c, _, _ in cases[:2]], dtype=np.uint32)
    assert [int(v) for v in philox4x32_10(ctrs, (0, 0))[0]] == list(cases[0][2])


def test_dropout_rule_host_side():
    """Threshold / scale of the library's fp32 evaluation, and the lane layout of one group."""
    assert dropout_threshold_scale(0.1) == (6554, float(np.float32(1) / np.float32(0.9)))
    assert dropout_threshold_scale(0.5) == (32768, 2.0)
    assert dropout_threshold_scale(1e-9)[0] == 1
    keep = dropout_keep(16, 0.5, 0x0123456789ABCDEF, 3)
    w = philox4x32_10(np.array([[1, 0, 3, 0x0B200B00]], np.uint32), (0x89ABCDEF, 0x01234567))[0]
    want = [((int(w[e // 2]) >> (16 * (e % 2))) & 0xFFFF) >= 32768 for e in range(8)]
    assert list(keep[8:]) == want
    rate = dropout_keep(1 << 16, 0.1, 5, 1).mean()
    assert abs(rate - 0.9) < 0.01


# --------------------------------------------------------------------------------------------------------------------
# helpers
# --------------------------------------------------------------------------------------------------------------------
CONFIGS = [(1, 128), (1, 256), (2, 128), (2, 256), (0, 0)]          # (cta_group, block_n); 0/0 = automatic choice
MAJORS = [(0, 0), (0, 1), (1, 1)]                                    # KK, K.MN (dgrad form), MN.MN (wgrad form)
INSTANTIATIONS = [(am, bm, e) for am, bm in MAJORS for e in (EPI_BF16_BIAS, EPI_BF16_DGELU, EPI_F32)]
INSTANTIATIONS += [(0, 0, EPI_BF16_BIAS_GELU), (0, 0, EPI_F32_BIAS_RESID)]
TAIL_M = (1, 40, 129, 257, 2056)
TAIL_N = (8, 72, 264)
TAIL_K = (8, 72, 136, 2056)
# more tiles than CTA slots for every configuration (2.3 - 4.3 waves): both accumulator stages and the smem-stage
# phases wrap several times per CTA
MULTIWAVE = (2056, 4616, 200)


def _ops():
    from vlm_bridge_b200 import ops
    return ops


def _lib():
    from vlm_bridge_b200 import _lib as L
    return L


@contextlib.contextmanager
def _sm_limit(n: int):
    lib = _lib().lib()
    prev_limit, prev_dual = lib.b200b_get_sm_limit(), lib.b200b_gemm_set_dual(-1)
    try:
        lib.b200b_set_sm_limit(n)
        yield lib
    finally:
        lib.b200b_set_sm_limit(prev_limit)
        lib.b200b_gemm_set_dual(prev_dual)


def _ints(shape, g, lim=4):
    return torch.randint(-lim, lim + 1, shape, generator=g, device="cuda").float()


def _store(mat: torch.Tensor, pitched: bool, dtype=None) -> torch.Tensor:
    """A copy of 2-D `mat` as a view with unit inner stride and row pitch round_up(cols, 8) (+ 24 if pitched)."""
    rows, cols = mat.shape
    ld = -(-cols // 8) * 8 + (24 if pitched else 0)
    buf = torch.zeros(rows, ld, device="cuda", dtype=dtype or mat.dtype)
    buf[:, :cols] = mat
    return buf[:, :cols]


_GUARD_ROWS, _EXTRA_ROWS = 2, 3
_SENTINEL = {torch.bfloat16: (torch.int16, 0x7FA5), torch.float32: (torch.int32, 0x7FC01234)}   # NaN payloads


def _sentinel_view(m, n, dtype, pitched):
    """(buffer, view [m, n] of it, window mask): guard rows before the base, 24 spare columns inside the pitch when
    pitched, rows below m; the whole buffer holds the sentinel bit pattern."""
    ld = n + (24 if pitched else 0)
    rows = _GUARD_ROWS + m + _EXTRA_ROWS
    buf = torch.empty(rows, ld, device="cuda", dtype=dtype)
    itype, bits = _SENTINEL[dtype]
    buf.view(itype).fill_(bits)
    win = torch.zeros(rows, ld, device="cuda", dtype=torch.bool)
    win[_GUARD_ROWS:_GUARD_ROWS + m, :n] = True
    return buf, buf[_GUARD_ROWS:_GUARD_ROWS + m, :n], win


def _sentinel_intact(buf, win) -> bool:
    itype, bits = _SENTINEL[buf.dtype]
    return bool((buf.view(itype)[~win] == bits).all())


def _bf16(x64: torch.Tensor) -> torch.Tensor:
    """fp64 values that are exact in fp32 -> bf16 with round-to-nearest-even."""
    return x64.float().bfloat16()


def _bf16_ulp(x: torch.Tensor) -> torch.Tensor:
    """ulp of bf16 at |x| (fp64), 2^-133 at zero."""
    _, e = torch.frexp(x.abs())
    ulp = torch.ldexp(torch.ones_like(x), e - 8).clamp_min(2.0 ** -133)
    return torch.where(x == 0, torch.full_like(x, 2.0 ** -133), ulp)


def _gelu64(x):
    return x * 0.5 * torch.special.erfc(-x / math.sqrt(2.0))


def _gelu_grad64(x):
    return 0.5 * torch.special.erfc(-x / math.sqrt(2.0)) + x * torch.exp(-0.5 * x * x) / math.sqrt(2.0 * math.pi)


# --------------------------------------------------------------------------------------------------------------------
# exact by construction: every built instantiation x tile configuration on tail shapes and one multi-wave shape
# --------------------------------------------------------------------------------------------------------------------
def _exact_case(am, bm, epi, m, n, k, cfg, i) -> list[str]:
    """Run one exact-integer GEMM; return the list of violated properties."""
    ops = _ops()
    pitched = i % 2 == 1
    use_bias = i % 3 != 2
    beta = (0.0, 0.5, 1.0)[i % 3]
    g = torch.Generator(device="cuda").manual_seed(7919 * i + 131 * epi + 17 * am + bm + 1)
    A, B = _ints((m, k), g), _ints((n, k), g)
    a = _store(A.t() if am else A, pitched, torch.bfloat16)
    b = _store(B.t() if bm else B, pitched, torch.bfloat16)
    acc = A.double() @ B.double().t()
    has_bias = epi in (EPI_BF16_BIAS, EPI_BF16_BIAS_GELU, EPI_F32_BIAS_RESID) and use_bias
    bias = (_ints((n,), g, 32) / 8) if has_bias else None
    bias64 = bias.double() if has_bias else 0.0
    out_dtype = torch.float32 if epi in (EPI_F32, EPI_F32_BIAS_RESID) else torch.bfloat16
    obuf, out, win = _sentinel_view(m, n, out_dtype, pitched)
    kw = dict(a_major=am, b_major=bm, epilogue=epi, out=out, bias=bias, cta_group=cfg[0], block_n=cfg[1])
    bad = []
    if epi == EPI_BF16_BIAS:
        ops.gemm(a, b, **kw)
        want = _bf16(acc + bias64)
    elif epi == EPI_F32:
        if beta == 0.0:       # out holds NaN (the sentinel): the kernel must not read it
            ops.gemm(a, b, **kw)
            want = acc.float()
        else:
            out0 = _ints((m, n), g, 32) / 8
            out.copy_(out0)
            ops.gemm(a, b, beta=beta, **kw)
            want = (beta * out0.double() + acc).float()
    elif epi == EPI_F32_BIAS_RESID:
        resid = _store(_ints((m, n), g, 32) / 8, pitched)
        ops.gemm(a, b, resid=resid, **kw)
        want = (resid.double() + _bf16(acc + bias64).double()).float()
    elif epi == EPI_BF16_BIAS_GELU:
        abuf, aux, awin = _sentinel_view(m, n, torch.bfloat16, not pitched)
        ops.gemm(a, b, aux=aux, **kw)
        want_aux = _bf16(acc + bias64)
        if not torch.equal(aux, want_aux):
            bad.append("aux != bf16(acc + bias)")
        if not _sentinel_intact(abuf, awin):
            bad.append("aux written out of bounds")
        ref = _gelu64(aux.double())
        bound = _bf16_ulp(ref) + 1e-6 * float(ref.abs().max())
        if not bool(((out.double() - ref).abs() <= bound).all()):
            bad.append("gelu(aux) beyond 1 bf16 ulp")
        want = None
    else:  # EPI_BF16_DGELU: u in {-16, +16}, where the kernel's gelu'(u) is exactly 0 / 1
        u = _store((torch.randint(0, 2, (m, n), generator=g, device="cuda").float() * 32 - 16), pitched,
                   torch.bfloat16)
        ops.gemm(a, b, aux=u, **kw)
        want = torch.where(u > 0, _bf16(acc), torch.zeros((), device="cuda", dtype=torch.bfloat16))
    if want is not None and not torch.equal(out, want):
        nbad = int((out.float() != want.float()).sum())
        bad.append(f"{nbad} of {m * n} outputs differ from the exact result")
    if not _sentinel_intact(obuf, win):
        bad.append("out written out of bounds")
    return [f"m={m} n={n} k={k} pitched={pitched} bias={has_bias} beta={beta}: {s}" for s in bad]


def _exact_shapes():
    shapes = [(m, n, TAIL_K[i % 4]) for i, (m, n) in enumerate((m, n) for m in TAIL_M for n in TAIL_N)]
    return shapes + [MULTIWAVE]


@gpu
@pytest.mark.parametrize("cfg", CONFIGS, ids=lambda c: f"cg{c[0]}_bn{c[1]}")
@pytest.mark.parametrize("am,bm,epi", INSTANTIATIONS, ids=[f"a{a}b{b}_{EPI_NAMES[e]}" for a, b, e in INSTANTIATIONS])
def test_gemm_exact_every_instantiation(am, bm, epi, cfg):
    fails = []
    for i, (m, n, k) in enumerate(_exact_shapes()):
        fails += _exact_case(am, bm, epi, m, n, k, cfg, i)
    torch.cuda.synchronize()
    assert not fails, "\n".join(fails[:12])


@gpu
@pytest.mark.parametrize("cfg", [(2, 128), (2, 256)], ids=lambda c: f"cg{c[0]}_bn{c[1]}")
def test_gemm_pair_with_empty_second_cta(cfg):
    """M <= 128 on CTA pairs: the odd CTA of every pair has no valid row (TMA zero-fill, all stores masked)."""
    fails = []
    for i, m in enumerate((1, 8, 100, 128)):
        for am, bm, epi in INSTANTIATIONS:
            fails += _exact_case(am, bm, epi, m, 264, 200, cfg, i + 3)
    assert not fails, "\n".join(fails[:12])


# --------------------------------------------------------------------------------------------------------------------
# realistic operands at bridge sizes: elementwise bounds, the measured ratio to the bound is printed
# --------------------------------------------------------------------------------------------------------------------
REALISTIC = [
    ("kk_bias_qproj", 0, 0, EPI_BF16_BIAS, 1024, 2304, 2304),
    ("kk_gelu_ffn_up", 0, 0, EPI_BF16_BIAS_GELU, 1024, 9216, 2304),
    ("kk_resid_ffn_down", 0, 0, EPI_F32_BIAS_RESID, 1024, 2304, 9216),
    ("kmn_dgrad", 0, 1, EPI_BF16_BIAS, 1024, 2304, 9216),
    ("kmn_dgelu", 0, 1, EPI_BF16_DGELU, 1024, 9216, 2304),
    ("mnmn_wgrad", 1, 1, EPI_F32, 2304, 2304, 1024),
    ("mnmn_wgrad_vision", 1, 1, EPI_F32, 4608, 1024, 2056),
    ("mnmn_wgrad_bf16", 1, 1, EPI_BF16_BIAS, 2304, 9216, 1024),
]


@gpu
@pytest.mark.parametrize("name,am,bm,epi,m,n,k", REALISTIC, ids=[c[0] for c in REALISTIC])
def test_gemm_realistic_elementwise_bound(name, am, bm, epi, m, n, k):
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(m + n + k + epi)
    A = (torch.randn(m, k, generator=g, device="cuda") * 0.5).bfloat16()
    B = (torch.randn(n, k, generator=g, device="cuda") * 0.02).bfloat16()
    a = A.t().contiguous() if am else A
    b = B.t().contiguous() if bm else B
    A64, B64 = A.double(), B.double()
    acc = A64 @ B64.t()
    accb = 4.0 * math.sqrt(k) * 2.0 ** -24 * (A64.abs() @ B64.abs().t())
    bias = torch.randn(n, generator=g, device="cuda") * 0.1
    ratios = {}

    def ratio(err, bound):
        return float((err / bound).max())

    if epi == EPI_BF16_BIAS:
        bias = bias if am == 0 and bm == 0 else None
        out = ops.gemm(a, b, a_major=am, b_major=bm, epilogue=epi, bias=bias)
        ref = acc + (bias.double() if bias is not None else 0.0)
        ratios["out"] = ratio((out.double() - ref).abs(), 1.01 * accb + (2.0 ** -8 + 2.0 ** -22) * ref.abs())
    elif epi == EPI_F32:
        out = ops.gemm(a, b, a_major=am, b_major=bm, epilogue=epi)
        ratios["acc"] = ratio((out.double() - acc).abs(), accb)
    elif epi == EPI_F32_BIAS_RESID:
        resid = torch.randn(m, n, generator=g, device="cuda")
        out = ops.gemm(a, b, epilogue=epi, bias=bias, resid=resid)
        y = acc + bias.double()
        ref = resid.double() + y
        bound = 1.01 * accb + (2.0 ** -8 + 2.0 ** -22) * y.abs() + 2.0 ** -23 * ref.abs()
        ratios["out"] = ratio((out.double() - ref).abs(), bound)
    elif epi == EPI_BF16_BIAS_GELU:
        out, aux = ops.gemm(a, b, epilogue=epi, bias=bias)
        u = acc + bias.double()
        ratios["aux"] = ratio((aux.double() - u).abs(), 1.01 * accb + (2.0 ** -8 + 2.0 ** -22) * u.abs())
        ref = _gelu64(aux.double())
        ratios["gelu"] = ratio((out.double() - ref).abs(), _bf16_ulp(ref) + 1e-6 * float(ref.abs().max()))
    else:  # EPI_BF16_DGELU
        u = torch.randn(m, n, generator=g, device="cuda").bfloat16()
        out = ops.gemm(a, b, a_major=am, b_major=bm, epilogue=epi, aux=u)
        gp = _gelu_grad64(u.double())
        ref = acc * gp
        bound = gp.abs() * (1.01 * accb + 2.0 ** -8 * acc.abs()) + _bf16_ulp(ref) + 1e-6 * float(ref.abs().max())
        ratios["dgelu"] = ratio((out.double() - ref).abs(), bound)
    torch.cuda.synchronize()
    print(f"[gemm bound ratio] {name}: " + ", ".join(f"{key} {v:.3f}" for key, v in ratios.items()))
    for key, v in ratios.items():
        assert v <= 1.0, f"{name}: {key} error is {v:.3f} x the bound"


# --------------------------------------------------------------------------------------------------------------------
# dropout, bit for bit
# --------------------------------------------------------------------------------------------------------------------
SEED = 0x9E3779B97F4A7C15      # both 32-bit halves of the key matter
DROP_STREAM = 7
DM, DN, DK = 300, 264, 72      # m * n not a multiple of any tile; k one full and one partial k block


def _keep_tensor(m, n, p, seed=SEED, stream=DROP_STREAM):
    return torch.from_numpy(dropout_keep(m * n, p, seed, stream).reshape(m, n)).cuda()


def _seed_tensor(seed):
    return torch.tensor([seed - (1 << 64) if seed >= 1 << 63 else seed], dtype=torch.int64, device="cuda")


@gpu
@pytest.mark.parametrize("p", [0.1, 0.5])
def test_dropout_masks_exact(p):
    """GELU / residual / dGELU epilogues and cast_bf16 / cast_bf16_colsum apply exactly the host Philox mask of
    (seed, stream, row * n + col), whatever the tile configuration, SM limit or output pitch; a seed read from a
    device pointer gives the same result as the value passed directly."""
    ops = _ops()
    thr, scale = dropout_threshold_scale(p)
    keep = _keep_tensor(DM, DN, p)
    zero = torch.zeros((), device="cuda", dtype=torch.bfloat16)
    g = torch.Generator(device="cuda").manual_seed(int(p * 1000))
    A = _ints((DM, DK), g).bfloat16()
    W = _ints((DN, DK), g).bfloat16()
    acc = A.double() @ W.double().t()
    bias = _ints((DN,), g, 32) / 8
    drop = dict(dropout_p=p, seed=SEED, dropout_stream=DROP_STREAM)
    seed_t = _seed_tensor(SEED)
    indirect = dict(dropout_p=p, seed=seed_t.data_ptr(), dropout_stream=DROP_STREAM | SEED_INDIRECT)

    # GELU: the kept value is bf16(bf16(gelu(u)) * scale); the undropped output gives the kernel's bf16(gelu(u))
    h0, u0 = ops.gemm(A, W, epilogue=EPI_BF16_BIAS_GELU, bias=bias)
    want_gelu = torch.where(keep, (h0.float() * scale).bfloat16(), zero)
    assert torch.equal(u0, _bf16(acc + bias.double()))
    fails = []
    for limit in (0, 16):
        with _sm_limit(limit):
            for j, (cg, bn) in enumerate(CONFIGS):
                pitched = j % 2 == 1
                obuf, out, win = _sentinel_view(DM, DN, torch.bfloat16, pitched)
                _, aux, _ = _sentinel_view(DM, DN, torch.bfloat16, not pitched)
                ops.gemm(A, W, epilogue=EPI_BF16_BIAS_GELU, bias=bias, out=out, aux=aux, cta_group=cg, block_n=bn,
                         **drop)
                if not (torch.equal(out, want_gelu) and torch.equal(aux, u0) and _sentinel_intact(obuf, win)):
                    fails.append(f"gelu limit={limit} cg={cg} bn={bn} pitched={pitched}")
    assert not fails, fails
    out_ind, _ = ops.gemm(A, W, epilogue=EPI_BF16_BIAS_GELU, bias=bias, **indirect)
    assert torch.equal(out_ind, want_gelu), "gemm: indirect seed differs from the direct one"

    # residual: resid + (bf16(bf16(acc + bias) * scale) or 0)
    resid = _ints((DM, DN), g, 32) / 8
    y = _bf16(acc + bias.double()).float()
    want_resid = resid + torch.where(keep, (y * scale).bfloat16().float(), torch.zeros((), device="cuda"))
    for cg, bn in CONFIGS:
        out = ops.gemm(A, W, epilogue=EPI_F32_BIAS_RESID, bias=bias, resid=resid, cta_group=cg, block_n=bn, **drop)
        assert torch.equal(out, want_resid), f"resid cg={cg} bn={bn}"

    # dGELU (dgrad form, B stored [K, N]): u = +-16 makes the kernel's gelu'(u) exactly 1 / 0
    u = (torch.randint(0, 2, (DM, DN), generator=g, device="cuda").float() * 32 - 16).bfloat16()
    d = torch.where(keep, (_bf16(acc).float() * scale).bfloat16(), zero)
    want_dgelu = torch.where(u > 0, d, zero)
    Wt = W.t().contiguous()
    for cg, bn in CONFIGS:
        out = ops.gemm(A, Wt, b_major=1, epilogue=EPI_BF16_DGELU, aux=u, cta_group=cg, block_n=bn, **drop)
        assert torch.equal(out, want_dgelu), f"dgelu cg={cg} bn={bn}"

    # the dropout-backward casts draw the same mask over a contiguous [m, n]
    x = torch.randn(DM, DN, generator=g, device="cuda")
    want_cast = torch.where(keep, (x.bfloat16().float() * scale).bfloat16(), zero)
    assert torch.equal(ops.cast_bf16(x, **drop), want_cast)
    assert torch.equal(ops.cast_bf16(x, **indirect), want_cast), "cast_bf16: indirect seed"
    yc, cs = ops.cast_bf16_colsum(x, **drop)
    assert torch.equal(yc, want_cast)
    yc2, cs2 = ops.cast_bf16_colsum(x, **indirect)
    assert torch.equal(yc2, want_cast) and torch.equal(cs2, cs), "cast_bf16_colsum: indirect seed"
    ref = want_cast.double().sum(0)
    assert bool(((cs.double() - ref).abs() <= DM * 2.0 ** -24 * want_cast.double().abs().sum(0)).all())
    assert thr > 0 and abs(float(keep.float().mean()) - (1 - p)) < 0.02


@gpu
def test_dropout_non_finite_values():
    """A kept inf / NaN propagates; a dropped position is an exact 0 whatever its value (b200_bridge.h, Dropout)."""
    ops = _ops()
    p = 0.5
    keep = _keep_tensor(DM, DN, p)
    g = torch.Generator(device="cuda").manual_seed(11)
    A = _ints((DM, DK), g).bfloat16()
    W = _ints((DN, DK), g).bfloat16()
    bias = _ints((DN,), g, 32) / 8
    special = torch.tensor([math.inf, -math.inf, math.nan], device="cuda")
    bias[:3] = special
    drop = dict(dropout_p=p, seed=SEED, dropout_stream=DROP_STREAM)
    cols = slice(0, 3)

    h, _ = ops.gemm(A, W, epilogue=EPI_BF16_BIAS_GELU, bias=bias, **drop)
    hs, ks = h[:, cols].float(), keep[:, cols]
    assert bool((hs[~ks] == 0).all()), "gelu: dropped non-finite value is not 0"
    assert not bool(torch.isfinite(hs[ks]).any()), "gelu: kept non-finite value became finite"
    assert bool((h[:, 0].float()[keep[:, 0]] == math.inf).all())           # gelu(+inf) = +inf

    resid = torch.randn(DM, DN, generator=g, device="cuda")
    o = ops.gemm(A, W, epilogue=EPI_F32_BIAS_RESID, bias=bias, resid=resid, **drop)
    assert torch.equal(o[:, cols][~ks], resid[:, cols][~ks]), "resid: dropped non-finite value added something"
    assert not bool(torch.isfinite(o[:, cols][ks]).any())
    o0 = ops.gemm(A, W, epilogue=EPI_F32_BIAS_RESID, bias=bias, resid=resid)
    assert not bool(torch.isfinite(o0[:, cols]).any()), "resid: non-finite value lost without dropout"

    # dGELU multiplies the (possibly dropped) gradient by gelu'(aux): a non-finite aux gives NaN everywhere
    u = torch.randn(DM, DN, generator=g, device="cuda").bfloat16()
    u[:, :3] = special.bfloat16()
    o = ops.gemm(A, W.t().contiguous(), b_major=1, epilogue=EPI_BF16_DGELU, aux=u, **drop)
    assert bool(torch.isnan(o[:, cols].float()).all())
    assert bool(torch.isfinite(o[:, 3:].float()).all())

    x = torch.randn(DM, DN, generator=g, device="cuda")
    x[:, :3] = special
    y = ops.cast_bf16(x, **drop)
    assert bool((y[:, cols].float()[~ks] == 0).all()), "cast_bf16: dropped non-finite value is not 0"
    assert not bool(torch.isfinite(y[:, cols].float()[ks]).any())
    y0 = ops.cast_bf16(x)
    assert torch.equal(torch.isnan(y0.float()), torch.isnan(x)) and torch.equal(torch.isinf(y0.float()), torch.isinf(x))


# --------------------------------------------------------------------------------------------------------------------
# scheduling: the result does not depend on the SM limit or on the tile configuration
# --------------------------------------------------------------------------------------------------------------------
LIMITS = [0, 1, 2, 3, 16, 147]


@gpu
@pytest.mark.parametrize("am,bm,epi", INSTANTIATIONS, ids=[f"a{a}b{b}_{EPI_NAMES[e]}" for a, b, e in INSTANTIATIONS])
def test_gemm_bit_identical_across_sm_limits_and_tiles(am, bm, epi):
    """Realistic operands, one shape, every SM limit (1 included: no CTA pair fits, single CTAs run) x every tile
    configuration: the per-element k order is the same everywhere, so every output is bit-identical."""
    ops = _ops()
    m, n, k = 1040, 1032, 264
    g = torch.Generator(device="cuda").manual_seed(99 + epi)
    A = (torch.randn(m, k, generator=g, device="cuda") * 0.5).bfloat16()
    B = (torch.randn(n, k, generator=g, device="cuda") * 0.02).bfloat16()
    a = A.t().contiguous() if am else A
    b = B.t().contiguous() if bm else B
    kw = dict(a_major=am, b_major=bm, epilogue=epi)
    if epi in (EPI_BF16_BIAS_GELU, EPI_F32_BIAS_RESID):
        kw.update(bias=torch.randn(n, generator=g, device="cuda"), dropout_p=0.1, seed=5, dropout_stream=2)
    if epi == EPI_F32_BIAS_RESID:
        kw["resid"] = torch.randn(m, n, generator=g, device="cuda")
    if epi == EPI_BF16_DGELU:
        kw["aux"] = torch.randn(m, n, generator=g, device="cuda").bfloat16()

    def run(cfg):
        r = ops.gemm(a, b, cta_group=cfg[0], block_n=cfg[1], **kw)
        return r[0] if isinstance(r, tuple) else r

    base = run((0, 0))
    torch.cuda.synchronize()
    assert not bool(torch.isnan(base.float()).any())
    diffs = []
    for limit in LIMITS:
        with _sm_limit(limit):
            for cfg in CONFIGS:
                if not torch.equal(run(cfg), base):
                    diffs.append(f"limit={limit} cg={cfg[0]} bn={cfg[1]}")
    torch.cuda.synchronize()
    assert not diffs, diffs


@gpu
def test_grouped_launch_under_sm_limits():
    """b200b_gemm_dual: under a limit of 1 (no CTA pair fits) it runs its two launches; every limit gives the
    result of the unlimited grouped launch."""
    ops, L = _ops(), _lib()
    g = torch.Generator(device="cuda").manual_seed(3)
    dy = (torch.randn(1024, 2304, generator=g, device="cuda") * 0.5).bfloat16()
    w = (torch.randn(2304, 2304, generator=g, device="cuda") * 0.02).bfloat16()
    x = (torch.randn(1024, 2304, generator=g, device="cuda") * 0.5).bfloat16()
    with _sm_limit(0) as lib:
        lib.b200b_gemm_set_dual(1)
        dx0, dw0 = ops.gemm_grad_pair(dy, w, x)
    for limit in (1, 2, 16):
        with _sm_limit(limit) as lib:
            lib.b200b_gemm_set_dual(1)
            before = L.launch_count()
            dx, dw = ops.gemm_grad_pair(dy, w, x)
            launches = L.launch_count() - before
        assert torch.equal(dx, dx0) and torch.equal(dw, dw0), f"limit {limit}"
        # with few pairs the tile choice prefers 256-wide tiles, which the grouped kernel does not cover
        assert launches == 2 if limit == 1 else launches in (1, 2), f"limit {limit}: {launches} launches"


# --------------------------------------------------------------------------------------------------------------------
# argument checks: documented code, a message, nothing launched
# --------------------------------------------------------------------------------------------------------------------
@gpu
def test_gemm_argument_checks():
    L = _lib()
    lib = L.lib()
    dev = "cuda"
    n = 128
    a = torch.zeros(n, n + 8, device=dev, dtype=torch.bfloat16)
    b = torch.zeros(n, n, device=dev, dtype=torch.bfloat16)
    o16 = torch.zeros(n, n, device=dev, dtype=torch.bfloat16)
    o32 = torch.zeros(n, n + 8, device=dev, dtype=torch.float32)
    aux = torch.zeros(n, n, device=dev, dtype=torch.bfloat16)
    resid = torch.zeros(n, n, device=dev, dtype=torch.float32)

    def args(**kw):
        base = dict(a=a.data_ptr(), b=b.data_ptr(), a_major=0, b_major=0, m=n, n=n, k=n, lda=n + 8, ldb=n,
                    epilogue=EPI_BF16_BIAS, block_n=0, out=o16.data_ptr(), ldo=n, aux=None, ldaux=0, bias=None,
                    resid=None, ldr=0, beta=0.0, dropout_p=0.0, seed=0, dropout_stream=0, cta_group=0)
        base.update(kw)
        return L.GemmArgs(**base)

    f32 = dict(epilogue=EPI_F32, out=o32.data_ptr(), ldo=n + 8)
    cases = [
        ("a_major=1, b_major=0", dict(a_major=1, b_major=0), ERR_ARG, "a_major=1"),
        ("n % 8 != 0", dict(n=124), ERR_SHAPE, "multiple of 8"),
        ("m == 0", dict(m=0), ERR_SHAPE, "m,n,k > 0"),
        ("misaligned a", dict(a=a.data_ptr() + 2), ERR_ALIGN, "aligned"),
        ("misaligned out", dict(out=o16.data_ptr() + 8), ERR_ALIGN, "aligned"),
        ("lda % 8", dict(lda=n + 4), ERR_ALIGN, "aligned"),
        ("ldb % 8", dict(ldb=n - 2), ERR_ALIGN, "aligned"),
        ("f32 ldo % 4", dict(f32, ldo=n + 2), ERR_ALIGN, "aligned"),
        ("misaligned bias", dict(bias=resid.data_ptr() + 4), ERR_ALIGN, "bias"),
        ("dropout_p = 1", dict(dropout_p=1.0), ERR_ARG, "dropout_p"),
        ("dropout_p < 0", dict(dropout_p=-0.1), ERR_ARG, "dropout_p"),
        ("dropout_p NaN", dict(dropout_p=math.nan), ERR_ARG, "dropout_p"),
        ("gelu without aux", dict(epilogue=EPI_BF16_BIAS_GELU), ERR_ARG, "aux"),
        ("dgelu without aux", dict(epilogue=EPI_BF16_DGELU), ERR_ARG, "aux"),
        ("dgelu aux pitch", dict(epilogue=EPI_BF16_DGELU, aux=aux.data_ptr(), ldaux=n - 4), ERR_ARG, "aux"),
        ("resid without resid", dict(f32, epilogue=EPI_F32_BIAS_RESID), ERR_ARG, "resid"),
        ("gelu, MN-major b", dict(epilogue=EPI_BF16_BIAS_GELU, aux=aux.data_ptr(), ldaux=n, b_major=1), ERR_ARG,
         "not built"),
        ("gelu, MN-major a and b", dict(epilogue=EPI_BF16_BIAS_GELU, aux=aux.data_ptr(), ldaux=n, a_major=1,
                                        b_major=1), ERR_ARG, "not built"),
        ("resid, MN-major b", dict(f32, epilogue=EPI_F32_BIAS_RESID, resid=resid.data_ptr(), ldr=n, b_major=1),
         ERR_ARG, "not built"),
        ("resid, MN-major a and b", dict(f32, epilogue=EPI_F32_BIAS_RESID, resid=resid.data_ptr(), ldr=n, a_major=1,
                                         b_major=1), ERR_ARG, "not built"),
        ("unknown epilogue", dict(epilogue=5), ERR_ARG, "epilogue"),
        ("block_n 64", dict(block_n=64), ERR_ARG, "block_n"),
        ("cta_group 3", dict(cta_group=3), ERR_ARG, "cta_group"),
    ]
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for what, kw, code, word in cases:
        before = L.launch_count()
        rc = lib.b200b_gemm(C.byref(args(**kw)), stream)
        msg = lib.b200b_last_error().decode()
        assert rc == code, f"{what}: rc {rc}, expected {code} ({msg})"
        assert word in msg, f"{what}: message {msg!r}"
        assert L.launch_count() == before, f"{what}: launched a kernel"
    # the same arguments without the fault do run
    assert lib.b200b_gemm(C.byref(args()), stream) == 0
    torch.cuda.synchronize()
