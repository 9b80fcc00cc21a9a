"""Op-level parity of the row kernels (csrc/elementwise.cu) against float64 references.

LayerNorm statistics are held to a few fp32 ulps of the fp64 statistics of the same fp32 input, y to one bf16 ulp of
the fp64 formula; the LayerNorm input gradient to fp32 rounding of its terms plus the summation error of its two row
means; column sums to rows * 2^-24 * sum|terms|. Casts are bit-exact: cast_bf16 against torch's round-to-nearest-even
(signed zeros, subnormals, overflow to inf, inf and NaN included), bf16_to_f32 against one fp32 multiply.

Shapes sit on every dispatch boundary of the kernels (the warp kernel's float4-per-lane count NV, the row kernel's
float4-per-thread count VPT, the cast kernel's groups-per-thread GPT) and row counts straddle 2 x SMs and 8 x SMs,
where the row loops start striding over the grid.

The last test feeds each kernel's output straight into the next library kernel on one stream with no
synchronisation (programmatic dependent launch on) and compares with the same chain synchronised after every step
and with a run in a subprocess where programmatic dependent launch is off: all bit-identical.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu
U = 2.0 ** -24
EPS = float(np.float32(1e-5))        # the kernels add eps in fp32

ROWS = (1, 7, 295, 296, 297, 1185, 2056)                      # around 2 x 148 and 8 x 148 SMs, and above them
# warp kernel: NV = ceil(dim / 128) float4 per lane, built for NV in {1, 2, 4, 8, 18, 32}
WARP_DIMS = (4, 128, 132, 256, 260, 512, 516, 1000, 1024, 1028, 2304, 2308, 4096)
# row kernel: VPT = ceil(dim / 4 / 192) float4 per thread, built for VPT in {1, 2, 3, 6}
ROW_DIMS = (4, 768, 772, 1000, 1536, 1540, 2304, 2308, 4608)


def _ops():
    from vlm_bridge_b200 import ops
    return ops


def _lib():
    from vlm_bridge_b200 import _lib as L
    return L


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _bf16_ulp(x: torch.Tensor) -> torch.Tensor:
    _, e = torch.frexp(x.abs())
    ulp = torch.ldexp(torch.ones_like(x), e - 8).clamp_min(2.0 ** -133)
    return torch.where(x == 0, torch.full_like(x, 2.0 ** -133), ulp)


def _ln_input(rows: int, dim: int, seed: int) -> torch.Tensor:
    """Rows of four kinds: N(0.5, 2^2); constant rows (variance 0, sums exact); mean / std of 10, 100 or 1000;
    N(0, 1e-3^2) (variance below eps)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(rows, dim, generator=g, device="cuda")
    r = torch.arange(rows, device="cuda")
    kind = r % 4
    const = torch.tensor([0.0, 3.0, -2.5, 1024.0], device="cuda")[(r // 4) % 4]
    offset = torch.tensor([10.0, 100.0, 1000.0], device="cuda")[(r // 4) % 3]
    x = torch.where((kind == 0)[:, None], x * 2 + 0.5, x)
    x = torch.where((kind == 1)[:, None], const[:, None].expand(rows, dim), x)
    x = torch.where((kind == 2)[:, None], x + offset[:, None], x)
    x = torch.where((kind == 3)[:, None], x * 1e-3, x)
    return x.contiguous()


def _affine(dim, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    gamma = torch.randn(dim, generator=g, device="cuda")
    beta = torch.randn(dim, generator=g, device="cuda").bfloat16().float()   # y of a constant row is exactly beta
    return gamma, beta


def _check_ln_fwd(fwd, x, gamma, beta, what) -> list[str]:
    rows, dim = x.shape
    y, mean, rstd = fwd(x, gamma, beta)
    x64 = x.double()
    mean64 = x64.mean(1)
    var64 = (x64 - mean64[:, None]).square().mean(1)
    rstd64 = 1.0 / torch.sqrt(var64 + EPS)
    bad = []
    dm = (mean.double() - mean64).abs()
    if not bool((dm <= 16 * U * x64.abs().mean(1) + U * mean64.abs()).all()):
        bad.append(f"mean off by {float((dm / (U * x64.abs().mean(1))).max()):.1f} ulp of mean|x|")
    dr = (rstd.double() - rstd64).abs() / rstd64
    if not bool((dr <= 16 * U).all()):
        bad.append(f"rstd off by {float(dr.max() / U):.1f} ulp")
    # y against the fp64 formula evaluated with the kernel's own statistics
    xg = (x64 - mean.double()[:, None]) * rstd.double()[:, None] * gamma.double()
    ref = xg + beta.double()
    err = (y.double() - ref).abs()
    if not bool((err <= _bf16_ulp(ref) + 4 * U * (xg.abs() + beta.double().abs())).all()):
        bad.append(f"y beyond 1 bf16 ulp ({float((err / _bf16_ulp(ref)).max()):.2f} ulp)")
    const = (x == x[:, :1]).all(1)
    if bool(const.any()):
        if not bool((y[const].float() == beta).all()):
            bad.append("constant row: y != beta")
        if not bool(((rstd[const].double() * EPS ** 0.5 - 1).abs() <= 4 * U).all()):
            bad.append("constant row: rstd != 1/sqrt(eps)")
    return [f"{what} rows={rows} dim={dim}: {s}" for s in bad]


@gpu
@pytest.mark.parametrize("kernel", ["warp", "rows"])
def test_layernorm_forward(kernel):
    ops = _ops()
    fwd = ops.layernorm_fwd if kernel == "warp" else ops.layernorm_fwd_rows
    dims = WARP_DIMS if kernel == "warp" else ROW_DIMS
    fails = []
    for dim in dims:
        gamma, beta = _affine(dim, dim)
        for rows in ROWS:
            fails += _check_ln_fwd(fwd, _ln_input(rows, dim, rows * 7 + dim), gamma, beta, kernel)
    assert not fails, "\n".join(fails[:12])


@gpu
def test_layernorm_forward_rejects_unsupported_dims():
    ops = _ops()
    for fwd, too_wide in ((ops.layernorm_fwd, 4100), (ops.layernorm_fwd_rows, 4612)):
        for dim in (too_wide, 6):
            x = torch.zeros(3, dim, device="cuda")
            with pytest.raises(RuntimeError, match=r"rc=-1\)"):
                fwd(x, torch.ones(dim, device="cuda"), torch.zeros(dim, device="cuda"))
    x = torch.zeros(3, 6, device="cuda")
    dy = torch.zeros(3, 6, device="cuda", dtype=torch.bfloat16)
    st = torch.ones(3, device="cuda")
    with pytest.raises(RuntimeError, match=r"rc=-1\)"):
        ops.layernorm_bwd(dy, x, st, st, torch.ones(6, device="cuda"))
    with pytest.raises(RuntimeError, match=r"rc=-1\)"):
        ops.layernorm_bwd_fused(dy, x, st, st, torch.ones(6, device="cuda"))


def _ln_bwd_ref(dy, x, mean, rstd, gamma, dres):
    """fp64 dx, the elementwise bound of the kernel's fp32 evaluation, xhat."""
    rs = rstd.double()[:, None]
    xh = (x.double() - mean.double()[:, None]) * rs
    g = dy.double() * gamma.double()
    m1 = g.mean(1, keepdim=True)
    m2 = (g * xh).mean(1, keepdim=True)
    dx = rs * (g - m1 - xh * m2)
    r = dres.double() if dres is not None else 0.0
    # fp32 rounding of every term, plus the error of the two row sums (tree of depth < 64)
    bound = rs * (4 * U * (g.abs() + m1.abs() + (xh * m2).abs()) +
                  64 * U * (g.abs().mean(1, keepdim=True) + xh.abs() * (g * xh).abs().mean(1, keepdim=True)))
    bound = bound + 2 * U * (dx + r).abs()
    return dx + r, bound, xh


def _bwd_inputs(rows, dim, seed):
    x = _ln_input(rows, dim, seed)
    gamma, beta = _affine(dim, seed + 1)
    _, mean, rstd = _ops().layernorm_fwd_rows(x, gamma, beta)
    g = torch.Generator(device="cuda").manual_seed(seed + 2)
    dy = torch.randn(rows, dim, generator=g, device="cuda").bfloat16()
    dres = torch.randn(rows, dim, generator=g, device="cuda")
    return x, gamma, mean, rstd, dy, dres


def _colsum_ok(got, terms, rows_extra=0) -> bool:
    rows = terms.shape[0]
    ref = terms.sum(0)
    return bool(((got.double() - ref).abs() <= (rows + rows_extra) * U * terms.abs().sum(0)).all())


@gpu
def test_layernorm_backward_warp():
    ops = _ops()
    fails = []
    for dim in (4, 128, 260, 1000, 2304, 4096):
        for rows in (1, 7, 297, 1185, 2056):
            x, gamma, mean, rstd, dy, dres = _bwd_inputs(rows, dim, rows + 3 * dim)
            for with_res in (False, True):
                d = dres if with_res else None
                dx = ops.layernorm_bwd(dy, x, mean, rstd, gamma, d)
                ref, bound, _ = _ln_bwd_ref(dy, x, mean, rstd, gamma, d)
                if not bool(((dx.double() - ref).abs() <= bound).all()):
                    fails.append(f"rows={rows} dim={dim} dres={with_res}: dx beyond bound "
                                 f"({float(((dx.double() - ref).abs() / bound).max()):.2f})")
            alias = dres.clone()
            ops.layernorm_bwd(dy, x, mean, rstd, gamma, alias, out=alias)
            if not torch.equal(alias, ops.layernorm_bwd(dy, x, mean, rstd, gamma, dres)):
                fails.append(f"rows={rows} dim={dim}: dx aliasing dres differs")
    assert not fails, "\n".join(fails[:12])


@gpu
def test_layernorm_backward_fused():
    ops, L = _ops(), _lib()
    fails = []
    for dim in (4, 768, 772, 1536, 2304, 2308, 4608):
        for rows in (1, 7, 297, 1185, 2056):
            x, gamma, mean, rstd, dy, dres = _bwd_inputs(rows, dim, 5 * rows + dim)
            tag = f"rows={rows} dim={dim}"
            for with_res in (False, True):
                d = dres if with_res else None
                dx, dyn, dbeta, dgamma, cs = ops.layernorm_bwd_fused(dy, x, mean, rstd, gamma, d)
                ref, bound, xh = _ln_bwd_ref(dy, x, mean, rstd, gamma, d)
                if not bool(((dx.double() - ref).abs() <= bound).all()):
                    fails.append(f"{tag} dres={with_res}: dx beyond bound")
                if not torch.equal(dyn, dx.bfloat16()):
                    fails.append(f"{tag}: dy_next != bf16(dx)")
                if not _colsum_ok(dbeta, dy.double()):
                    fails.append(f"{tag}: dbeta")
                # dy * xhat: xhat is rounded twice in fp32 before the product
                if not _colsum_ok(dgamma, dy.double() * xh, rows_extra=3):
                    fails.append(f"{tag}: dgamma")
                if not _colsum_ok(cs, dyn.double()):
                    fails.append(f"{tag}: colsum(dy_next)")
            # dx written over dres in place
            alias = dres.clone()
            chunks = L.lib().b200b_row_chunks(rows)
            part = torch.empty(chunks, 3, dim, device="cuda")
            dyn2 = torch.empty(rows, dim, device="cuda", dtype=torch.bfloat16)
            L.check(L.lib().b200b_layernorm_bwd_fused(dy.data_ptr(), x.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
                                                      gamma.data_ptr(), alias.data_ptr(), alias.data_ptr(),
                                                      dyn2.data_ptr(), part.data_ptr(), rows, dim, _stream()),
                    "layernorm_bwd_fused")
            if not torch.equal(alias, dx):
                fails.append(f"{tag}: dx aliasing dres differs")
            # no input gradient wanted: dbeta / dgamma still come out, bit-equal
            dx0, dyn0, db0, dg0, cs0 = ops.layernorm_bwd_fused(dy, x, mean, rstd, gamma, dres, want_dx=False)
            if dx0 is not None or dyn0 is not None or cs0 is not None:
                fails.append(f"{tag}: want_dx=False returned dx")
            if not (torch.equal(db0, dbeta) and torch.equal(dg0, dgamma)):
                fails.append(f"{tag}: want_dx=False changes dbeta / dgamma")
    assert not fails, "\n".join(fails[:12])


# --------------------------------------------------------------------------------------------------------------------
# column sums
# --------------------------------------------------------------------------------------------------------------------
@gpu
def test_colsum_plain_layernorm_and_two_stage():
    ops = _ops()
    fails = []
    for cols in (4, 132, 2304, 9216):
        for rows in (1, 7, 297, 2056):
            g = torch.Generator(device="cuda").manual_seed(rows * 31 + cols)
            buf = torch.randn(rows, cols + 24, generator=g, device="cuda").bfloat16()
            dy = buf[:, :cols]                       # pitched
            x = torch.randn(rows, cols, generator=g, device="cuda") * 3 + 1
            mean = x.mean(1)
            rstd = torch.rsqrt(x.var(1, unbiased=False) + EPS)
            tag = f"rows={rows} cols={cols}"
            s = ops.colsum(dy)
            if not _colsum_ok(s, dy.double()):
                fails.append(f"{tag}: colsum")
            s2, gs = ops.colsum(dy, x=x, mean=mean, rstd=rstd)
            xh = (x.double() - mean.double()[:, None]) * rstd.double()[:, None]
            if not (torch.equal(s2, s) and _colsum_ok(gs, dy.double() * xh, rows_extra=3)):
                fails.append(f"{tag}: LayerNorm-mode colsum")
            t = ops.colsum_two_stage(dy)
            if not _colsum_ok(t, dy.double()):
                fails.append(f"{tag}: two-stage colsum")
            if not (torch.equal(ops.colsum(dy), s) and torch.equal(ops.colsum_two_stage(dy), t)):
                fails.append(f"{tag}: not deterministic")
    assert not fails, "\n".join(fails[:12])


@gpu
def test_finalize_colsums_multi_task():
    """One launch over tasks of different widths: a block past a shorter task's columns writes nothing; 17 tasks
    are rejected; the result is deterministic."""
    ops = _ops()
    g = torch.Generator(device="cuda").manual_seed(4)
    specs = [(4, 1, 8), (132, 5, 136), (2304, 64, 3 * 2304), (520, 300, 520), (9216, 3, 9216)]  # cols, chunks, stride
    parts = [torch.randn(ch, st, generator=g, device="cuda") for _, ch, st in specs]
    outs = [torch.full((c + 128,), 7.25, device="cuda") for c, _, _ in specs]
    tasks = [(p, o, c, ch, st) for p, o, (c, ch, st) in zip(parts, outs, specs)]
    ops.finalize_colsums(tasks)
    first = [o.clone() for o in outs]
    ops.finalize_colsums(tasks)
    for p, o, f, (c, ch, st) in zip(parts, outs, first, specs):
        assert torch.equal(o, f), f"cols={c}: not deterministic"
        assert bool((o[c:] == 7.25).all()), f"cols={c}: wrote past its columns"
        assert _colsum_ok(o[:c], p[:, :c].double()), f"cols={c}: sum"
    many = [(parts[0], outs[0], 4, 1, 8)] * 17
    with pytest.raises(RuntimeError, match=r"rc=-3\)"):
        ops.finalize_colsums(many)
    ops.finalize_colsums(many[:16])         # 16 is the documented maximum


# --------------------------------------------------------------------------------------------------------------------
# casts
# --------------------------------------------------------------------------------------------------------------------
_BIG_N = 2 * 148 * 8 * 256 * 8 + 24         # more 8-element groups than the capped grid has threads: the loop strides


def _special_floats():
    f = torch.tensor([0.0, -0.0, 1e-40, -3e-39, 1.4e-45, -1.4e-45, 1.17549435e-38, 9.18e-41,
                      1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8, -(1.0 + 2.0 ** -8), 1.0 + 2.0 ** -8 + 2.0 ** -20,
                      3.3895313892515355e38, 3.3961e38, 3.4028234663852886e38, -3.4028234663852886e38,
                      float("inf"), float("-inf"), float("nan"), 65504.0, 2.0 ** -126, 2.0 ** -133, 2.0 ** -134,
                      2.0 ** -134 * 3], dtype=torch.float32)
    return torch.cat([f, torch.zeros((-len(f)) % 8)])


def _same_bf16(a: torch.Tensor, b: torch.Tensor) -> bool:
    na, nb = torch.isnan(a.float()), torch.isnan(b.float())
    return torch.equal(na, nb) and torch.equal(a.view(torch.int16)[~na], b.view(torch.int16)[~nb])


@gpu
def test_cast_bf16_is_round_to_nearest_even():
    ops = _ops()
    sp = _special_floats().cuda()
    assert _same_bf16(ops.cast_bf16(sp), sp.bfloat16())
    g = torch.Generator(device="cuda").manual_seed(8)
    mant = torch.rand(_BIG_N, generator=g, device="cuda") + 1.0
    expo = torch.randint(-149, 128, (_BIG_N,), generator=g, device="cuda")
    sign = torch.randint(0, 2, (_BIG_N,), generator=g, device="cuda") * 2 - 1
    x = torch.ldexp(mant * sign, expo).float()       # every binade, subnormals, overflow to inf
    x[: len(sp)] = sp
    assert _same_bf16(ops.cast_bf16(x), x.bfloat16())
    out = torch.empty(_BIG_N + 16, device="cuda", dtype=torch.bfloat16).fill_(5.0)
    ops.cast_bf16(x, out=out[:_BIG_N])
    assert bool((out[_BIG_N:].float() == 5.0).all())
    with pytest.raises(RuntimeError, match=r"rc=-1\)"):
        ops.cast_bf16(torch.zeros(12, device="cuda"))


@gpu
def test_cast_bf16_colsum_branches():
    """groups per thread 1 / 2 / 4 (dim <= 2304, <= 4608, <= 9216); dim 9224 and dim % 8 != 0 are rejected."""
    ops = _ops()
    fails = []
    for dim in (8, 2304, 2312, 4608, 4616, 9216):
        for rows in (1, 297, 1185):
            g = torch.Generator(device="cuda").manual_seed(dim + rows)
            x = torch.randn(rows, dim, generator=g, device="cuda") * 3
            y, s = ops.cast_bf16_colsum(x)
            if not _same_bf16(y, x.bfloat16()):
                fails.append(f"rows={rows} dim={dim}: cast")
            if not _colsum_ok(s, y.double()):
                fails.append(f"rows={rows} dim={dim}: column sums")
    assert not fails, fails
    for dim in (9224, 12):
        with pytest.raises(RuntimeError, match=r"rc=-1\)"):
            ops.cast_bf16_colsum(torch.zeros(3, dim, device="cuda"))


@gpu
@pytest.mark.parametrize("scale", [1.0, 0.5, 1.0 / 3.0, 3.7e-5, -2.0, 1e30])
def test_bf16_to_f32_exact(scale):
    L = _lib()
    g = torch.Generator(device="cuda").manual_seed(1)
    mant = torch.rand(_BIG_N, generator=g, device="cuda") + 1.0
    expo = torch.randint(-133, 128, (_BIG_N,), generator=g, device="cuda")
    x = torch.ldexp(mant, expo).float().bfloat16()
    x[:24] = _special_floats()[:24].bfloat16().cuda()
    s32 = float(np.float32(scale))
    out = torch.full((_BIG_N + 8,), 3.0, device="cuda")
    L.check(L.lib().b200b_bf16_to_f32(x.data_ptr(), out.data_ptr(), _BIG_N, s32, _stream()), "bf16_to_f32")
    want = x.float() * s32
    got = out[:_BIG_N]
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(got), nan)
    assert torch.equal(got[~nan].view(torch.int32), want[~nan].view(torch.int32))
    assert bool((out[_BIG_N:] == 3.0).all())


# --------------------------------------------------------------------------------------------------------------------
# a chain of library kernels on one stream, no synchronisation in between
# --------------------------------------------------------------------------------------------------------------------
def _chain(sync_each: bool = False) -> dict:
    """cast_bf16 -> gemm(F32_BIAS_RESID) -> layernorm_fwd_rows -> layernorm_bwd_fused (-> finalize_colsums), each
    reading the previous kernel's output."""
    ops = _ops()
    T, D = 1040, 2304
    g = torch.Generator(device="cuda").manual_seed(2024)
    w32 = torch.randn(D, D, generator=g, device="cuda") * 0.02
    a = (torch.randn(T, D, generator=g, device="cuda") * 0.5).bfloat16()
    bias = torch.randn(D, generator=g, device="cuda") * 0.1
    resid = torch.randn(T, D, generator=g, device="cuda")
    gamma = torch.randn(D, generator=g, device="cuda")
    beta = torch.randn(D, generator=g, device="cuda")
    torch.cuda.synchronize()
    step = torch.cuda.synchronize if sync_each else (lambda: None)
    w16 = ops.cast_bf16(w32)
    step()
    h = ops.gemm(a, w16, epilogue=ops.EPI_F32_BIAS_RESID, bias=bias, resid=resid, dropout_p=0.1, seed=77,
                 dropout_stream=4)
    step()
    y, mean, rstd = ops.layernorm_fwd_rows(h, gamma, beta)
    step()
    dx, dyn, dbeta, dgamma, cs = ops.layernorm_bwd_fused(y, h, mean, rstd, gamma, resid)
    torch.cuda.synchronize()
    return dict(w16=w16, h=h, y=y, mean=mean, rstd=rstd, dx=dx, dyn=dyn, dbeta=dbeta, dgamma=dgamma, cs=cs)


@gpu
def test_kernel_chain_without_synchronisation(tmp_path):
    free = _chain()
    synced = _chain(sync_each=True)
    for key in free:
        assert torch.equal(free[key], synced[key]), f"{key}: differs from the synchronised chain"
    path = tmp_path / "chain_nopdl.pt"
    env = dict(os.environ, B200B_PDL="0")
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--chain", str(path)], env=env,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    other = torch.load(path)
    for key in free:
        assert torch.equal(free[key].cpu(), other[key]), f"{key}: differs with programmatic dependent launch off"


if __name__ == "__main__":
    if "--chain" in sys.argv:
        sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        res = _chain()
        torch.save({k: v.cpu() for k, v in res.items()}, sys.argv[sys.argv.index("--chain") + 1])
