"""Thin torch-tensor wrappers over the C ABI (one function per exported kernel family).

torch supplies device memory and the current stream only; all arithmetic happens inside
libb200_bridge.so. Every wrapper validates devices/dtypes, then passes raw pointers.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import (EPI_BF16_BIAS, EPI_BF16_BIAS_GELU, EPI_BF16_DGELU, EPI_F32,  # noqa: F401
                   EPI_F32_BIAS_RESID)


def _stream_ptr() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t: torch.Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


def _need_cuda(*ts: torch.Tensor | None) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("b200 bridge kernels need CUDA tensors (there is no CPU fallback)")


def gemm(a: torch.Tensor, b: torch.Tensor, *, a_major: int = 0, b_major: int = 0,
         epilogue: int = EPI_BF16_BIAS, out: torch.Tensor | None = None,
         bias: torch.Tensor | None = None, aux: torch.Tensor | None = None,
         resid: torch.Tensor | None = None, beta: float = 0.0, dropout_p: float = 0.0,
         seed: int = 0, dropout_stream: int = 0, block_n: int = 0, cta_group: int = 0) -> torch.Tensor:
    """acc[m,n] = sum_k A(m,k) B(n,k) on tcgen05 tensor cores with a fused epilogue.

    a_major=0: a is [M,K]; a_major=1: a is [K,M]. b_major=0: b is [N,K]; b_major=1: b is [K,N].
    """
    _need_cuda(a, b, out, bias, aux, resid)
    if a.dtype != torch.bfloat16 or b.dtype != torch.bfloat16:
        raise RuntimeError("gemm operands must be bf16")
    if a.dim() != 2 or b.dim() != 2 or a.stride(1) != 1 or b.stride(1) != 1:
        raise RuntimeError("gemm operands must be 2-D with unit inner stride")
    m, k = (a.shape[1], a.shape[0]) if a_major else (a.shape[0], a.shape[1])
    n, kb = (b.shape[1], b.shape[0]) if b_major else (b.shape[0], b.shape[1])
    if k != kb:
        raise RuntimeError(f"gemm: contraction mismatch {k} vs {kb}")
    out_f32 = epilogue in (EPI_F32_BIAS_RESID, EPI_F32)
    if out is None:
        out = torch.empty((m, n), device=a.device, dtype=torch.float32 if out_f32 else torch.bfloat16)
    if out.dtype != (torch.float32 if out_f32 else torch.bfloat16) or out.shape != (m, n) or out.stride(1) != 1:
        raise RuntimeError("gemm: bad `out` tensor")
    if epilogue == EPI_BF16_BIAS_GELU and aux is None:
        aux = torch.empty((m, n), device=a.device, dtype=torch.bfloat16)
    args = _lib.GemmArgs(
        a=a.data_ptr(), b=b.data_ptr(), a_major=a_major, b_major=b_major, m=m, n=n, k=k,
        lda=a.stride(0), ldb=b.stride(0), epilogue=epilogue, block_n=block_n,
        out=out.data_ptr(), ldo=out.stride(0),
        aux=_ptr(aux), ldaux=0 if aux is None else aux.stride(0),
        bias=_ptr(bias), resid=_ptr(resid), ldr=0 if resid is None else resid.stride(0),
        beta=beta, dropout_p=dropout_p, seed=seed, dropout_stream=dropout_stream, cta_group=cta_group)
    _lib.check(_lib.lib().b200b_gemm(C.byref(args), _stream_ptr()), "gemm")
    if epilogue == EPI_BF16_BIAS_GELU:
        return out, aux
    return out


def layernorm_fwd(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5):
    """x f32 [rows, dim] -> (y bf16, mean f32[rows], rstd f32[rows])."""
    _need_cuda(x, gamma, beta)
    rows, dim = x.shape
    y = torch.empty((rows, dim), device=x.device, dtype=torch.bfloat16)
    mean = torch.empty(rows, device=x.device, dtype=torch.float32)
    rstd = torch.empty(rows, device=x.device, dtype=torch.float32)
    _lib.check(_lib.lib().b200b_layernorm_fwd(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), y.data_ptr(),
                                              mean.data_ptr(), rstd.data_ptr(), rows, dim, eps, _stream_ptr()),
               "layernorm_fwd")
    return y, mean, rstd


def layernorm_bwd(dy: torch.Tensor, x: torch.Tensor, mean: torch.Tensor, rstd: torch.Tensor,
                  gamma: torch.Tensor, dres: torch.Tensor | None = None, out: torch.Tensor | None = None):
    """dx f32 = dres + LN-backward(dy bf16)."""
    _need_cuda(dy, x, mean, rstd, gamma, dres, out)
    rows, dim = x.shape
    if out is None:
        out = torch.empty_like(x)
    _lib.check(_lib.lib().b200b_layernorm_bwd(dy.data_ptr(), x.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
                                              gamma.data_ptr(), _ptr(dres), out.data_ptr(), rows, dim,
                                              _stream_ptr()), "layernorm_bwd")
    return out


def layernorm_fwd_rows(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5):
    """CTA-per-row LayerNorm forward: x f32 [rows, dim] -> (y bf16, mean, rstd)."""
    _need_cuda(x, gamma, beta)
    rows, dim = x.shape
    y = torch.empty((rows, dim), device=x.device, dtype=torch.bfloat16)
    mean = torch.empty(rows, device=x.device, dtype=torch.float32)
    rstd = torch.empty(rows, device=x.device, dtype=torch.float32)
    _lib.check(_lib.lib().b200b_layernorm_fwd_rows(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), y.data_ptr(),
                                                   mean.data_ptr(), rstd.data_ptr(), rows, dim, eps, _stream_ptr()),
               "layernorm_fwd_rows")
    return y, mean, rstd


def finalize_colsums(tasks) -> None:
    """tasks: [(partials tensor (any view), out f32 [cols], cols, chunks, chunk_stride)] -> one launch."""
    arr = (_lib.ColsumTask * len(tasks))()
    for i, (part, out, cols, chunks, stride) in enumerate(tasks):
        arr[i] = _lib.ColsumTask(part.data_ptr(), out.data_ptr(), cols, chunks, stride)
    _lib.check(_lib.lib().b200b_colsum_finalize(arr, len(tasks), _stream_ptr()), "colsum_finalize")


def layernorm_bwd_fused(dy, x, mean, rstd, gamma, dres=None, want_dx=True, want_dy_next=True):
    """Fused LN backward: returns (dx f32 | None, dy_next bf16 | None, dbeta, dgamma, colsum(dy_next) | None)."""
    _need_cuda(dy, x, mean, rstd, gamma, dres)
    rows, dim = x.shape
    chunks = _lib.lib().b200b_row_chunks(rows)
    part = torch.empty((chunks, 3, dim), device=x.device, dtype=torch.float32)
    dx = torch.empty_like(x) if want_dx else None
    dyn = torch.empty((rows, dim), device=x.device, dtype=torch.bfloat16) if (want_dx and want_dy_next) else None
    _lib.check(_lib.lib().b200b_layernorm_bwd_fused(dy.data_ptr(), x.data_ptr(), mean.data_ptr(), rstd.data_ptr(),
                                                    gamma.data_ptr(), _ptr(dres), _ptr(dx), _ptr(dyn), part.data_ptr(),
                                                    rows, dim, _stream_ptr()), "layernorm_bwd_fused")
    outs = [torch.empty(dim, device=x.device, dtype=torch.float32) for _ in range(3)]
    n_out = 3 if dyn is not None else 2
    finalize_colsums([(part[0, j], outs[j], dim, chunks, 3 * dim) for j in range(n_out)])
    return dx, dyn, outs[0], outs[1], (outs[2] if dyn is not None else None)


def cast_bf16_colsum(x: torch.Tensor, dropout_p: float = 0.0, seed: int = 0, dropout_stream: int = 0):
    """x f32 [rows, dim] -> (bf16 copy with the dropout-backward mask, its column sums f32 [dim])."""
    _need_cuda(x)
    rows, dim = x.shape
    chunks = _lib.lib().b200b_row_chunks(rows)
    part = torch.empty((chunks, dim), device=x.device, dtype=torch.float32)
    out = torch.empty((rows, dim), device=x.device, dtype=torch.bfloat16)
    _lib.check(_lib.lib().b200b_cast_bf16_colsum(x.data_ptr(), out.data_ptr(), part.data_ptr(), rows, dim, dropout_p,
                                                 seed, dropout_stream, _stream_ptr()), "cast_bf16_colsum")
    s = torch.empty(dim, device=x.device, dtype=torch.float32)
    finalize_colsums([(part, s, dim, chunks, dim)])
    return out, s


def colsum_two_stage(dy: torch.Tensor) -> torch.Tensor:
    """b200b_colsum_partials + b200b_colsum_finalize (the path the block backward uses)."""
    _need_cuda(dy)
    rows, cols = dy.shape
    part = torch.empty((64, cols), device=dy.device, dtype=torch.float32)
    ch = C.c_int(0)
    _lib.check(_lib.lib().b200b_colsum_partials(dy.data_ptr(), dy.stride(0), rows, cols, part.data_ptr(), C.byref(ch),
                                                _stream_ptr()), "colsum_partials")
    s = torch.empty(cols, device=dy.device, dtype=torch.float32)
    finalize_colsums([(part, s, cols, ch.value, cols)])
    return s


def colsum(dy: torch.Tensor, *, x: torch.Tensor | None = None, mean: torch.Tensor | None = None,
           rstd: torch.Tensor | None = None, out_sum: torch.Tensor | None = None,
           out_gsum: torch.Tensor | None = None, workspace: torch.Tensor | None = None):
    """Column sums of dy bf16 [rows, cols] (and the LayerNorm dgamma sums when x is given)."""
    _need_cuda(dy, x, out_sum, out_gsum)
    rows, cols = dy.shape
    if out_sum is None:
        out_sum = torch.empty(cols, device=dy.device, dtype=torch.float32)
    if x is not None and out_gsum is None:
        out_gsum = torch.empty(cols, device=dy.device, dtype=torch.float32)
    nbytes = _lib.lib().b200b_colsum_workspace_bytes(rows, cols)
    if workspace is None:
        workspace = torch.empty(nbytes, device=dy.device, dtype=torch.uint8)
    _lib.check(_lib.lib().b200b_colsum(dy.data_ptr(), dy.stride(0), _ptr(x), _ptr(mean), _ptr(rstd),
                                       out_sum.data_ptr(), _ptr(out_gsum), rows, cols, workspace.data_ptr(),
                                       workspace.numel(), _stream_ptr()), "colsum")
    return (out_sum, out_gsum) if x is not None else out_sum


def cast_bf16(x: torch.Tensor, out: torch.Tensor | None = None, dropout_p: float = 0.0, seed: int = 0,
              dropout_stream: int = 0) -> torch.Tensor:
    _need_cuda(x, out)
    if not x.is_contiguous() or x.dtype != torch.float32:
        raise RuntimeError("cast_bf16 needs a contiguous fp32 tensor")
    if out is None:
        out = torch.empty(x.shape, device=x.device, dtype=torch.bfloat16)
    _lib.check(_lib.lib().b200b_cast_bf16(x.data_ptr(), out.data_ptr(), x.numel(), dropout_p, seed,
                                          dropout_stream, _stream_ptr()), "cast_bf16")
    return out


def _attn_args(q, k, v, o, lse, batch, heads, len_q, len_k, head_dim, dropout_p, seed, dropout_stream):
    return _lib.AttnArgs(q=q.data_ptr(), ldq=q.stride(0), k=k.data_ptr(), ldk=k.stride(0),
                         v=v.data_ptr(), ldv=v.stride(0), o=o.data_ptr(), ldo=o.stride(0),
                         lse=lse.data_ptr(), batch=batch, heads=heads, len_q=len_q, len_k=len_k,
                         head_dim=head_dim, dropout_p=dropout_p, seed=seed, dropout_stream=dropout_stream,
                         reserved=0)


def attention_fwd(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, *, batch: int, heads: int,
                  len_q: int, len_k: int, head_dim: int, dropout_p: float = 0.0, seed: int = 0,
                  dropout_stream: int = 0, out: torch.Tensor | None = None):
    """q: [batch*len_q, >=heads*head_dim] bf16 (2-D view, any row pitch); k, v: [batch*len_k, ...].

    Returns (o bf16 [batch*len_q, heads*head_dim], lse f32 [batch, heads, len_q])."""
    _need_cuda(q, k, v, out)
    if out is None:
        out = torch.empty((batch * len_q, heads * head_dim), device=q.device, dtype=torch.bfloat16)
    lse = torch.empty((batch, heads, len_q), device=q.device, dtype=torch.float32)
    args = _attn_args(q, k, v, out, lse, batch, heads, len_q, len_k, head_dim, dropout_p, seed, dropout_stream)
    _lib.check(_lib.lib().b200b_attention_fwd(C.byref(args), _stream_ptr()), "attention_fwd")
    return out, lse


def attention_bwd(d_o: torch.Tensor, q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, o: torch.Tensor,
                  lse: torch.Tensor, dq: torch.Tensor, dk: torch.Tensor, dv: torch.Tensor, *, batch: int,
                  heads: int, len_q: int, len_k: int, head_dim: int, dropout_p: float = 0.0, seed: int = 0,
                  dropout_stream: int = 0, workspace: torch.Tensor | None = None) -> None:
    """Writes dq / dk / dv (bf16 2-D views, any row pitch)."""
    _need_cuda(d_o, q, k, v, o, lse, dq, dk, dv)
    nbytes = _lib.lib().b200b_attention_bwd_workspace_bytes(batch, heads, len_q, len_k)
    if workspace is None:
        workspace = torch.empty(nbytes, device=q.device, dtype=torch.uint8)
    args = _attn_args(q, k, v, o, lse, batch, heads, len_q, len_k, head_dim, dropout_p, seed, dropout_stream)
    args.d_o, args.lddo = d_o.data_ptr(), d_o.stride(0)
    args.dq, args.lddq = dq.data_ptr(), dq.stride(0)
    args.dk, args.lddk = dk.data_ptr(), dk.stride(0)
    args.dv, args.lddv = dv.data_ptr(), dv.stride(0)
    args.workspace, args.workspace_bytes = workspace.data_ptr(), workspace.numel()
    _lib.check(_lib.lib().b200b_attention_bwd(C.byref(args), _stream_ptr()), "attention_bwd")


def kv_cache_pack(kv: torch.Tensor, *, batch: int, len_k: int, heads: int, head_dim: int,
                  num_blocks: int) -> torch.Tensor:
    """kv bf16 [batch*len_k, num_blocks*2*heads*head_dim] -> decode layout (flat uint8 tensor)."""
    _need_cuda(kv)
    nbytes = _lib.lib().b200b_kv_cache_packed_bytes(batch, len_k, heads, head_dim, num_blocks)
    packed = torch.empty(nbytes, device=kv.device, dtype=torch.uint8)
    _lib.check(_lib.lib().b200b_kv_cache_pack(kv.data_ptr(), kv.stride(0), packed.data_ptr(), batch, len_k, heads,
                                              head_dim, num_blocks, _stream_ptr()), "kv_cache_pack")
    return packed


def attention_decode_packed(q: torch.Tensor, kv_packed: torch.Tensor, *, block_index: int, num_blocks: int,
                            batch: int, heads: int, len_q: int, len_k: int, head_dim: int,
                            out: torch.Tensor | None = None, want_lse: bool = True):
    """Cross-attention of <= 64 query rows per image against block `block_index` of a packed K/V cache."""
    _need_cuda(q, kv_packed, out)
    if out is None:
        out = torch.empty((batch * len_q, heads * head_dim), device=q.device, dtype=torch.bfloat16)
    lse = torch.empty((batch, heads, len_q), device=q.device, dtype=torch.float32) if want_lse else None
    _lib.check(_lib.lib().b200b_attention_decode_packed(
        q.data_ptr(), q.stride(0), kv_packed.data_ptr(), block_index, num_blocks, out.data_ptr(), out.stride(0),
        _ptr(lse), batch, heads, len_q, len_k, head_dim, _stream_ptr()), "attention_decode_packed")
    return out, lse


def kv_cache_pack_tc(kv: torch.Tensor, *, batch: int, len_k: int, heads: int, head_dim: int,
                     num_blocks: int) -> torch.Tensor:
    """kv bf16 [batch*len_k, num_blocks*2*heads*head_dim] -> tcgen05 decode layout (flat uint8 tensor)."""
    _need_cuda(kv)
    nbytes = _lib.lib().b200b_kv_cache_tc_bytes(batch, len_k, heads, head_dim, num_blocks)
    packed = torch.empty(nbytes, device=kv.device, dtype=torch.uint8)
    _lib.check(_lib.lib().b200b_kv_cache_pack_tc(kv.data_ptr(), kv.stride(0), packed.data_ptr(), batch, len_k, heads,
                                                 head_dim, num_blocks, _stream_ptr()), "kv_cache_pack_tc")
    return packed


def attention_decode_tc(q: torch.Tensor, kv_tc: torch.Tensor, *, block_index: int, num_blocks: int, batch: int,
                        heads: int, len_q: int, len_k: int, head_dim: int, out: torch.Tensor | None = None,
                        want_lse: bool = True):
    """Cross-attention of <= 64 query rows per image against block `block_index` of a tc-packed K/V cache."""
    _need_cuda(q, kv_tc, out)
    if out is None:
        out = torch.empty((batch * len_q, heads * head_dim), device=q.device, dtype=torch.bfloat16)
    lse = torch.empty((batch, heads, len_q), device=q.device, dtype=torch.float32) if want_lse else None
    _lib.check(_lib.lib().b200b_attention_decode_tc(
        q.data_ptr(), q.stride(0), kv_tc.data_ptr(), block_index, num_blocks, out.data_ptr(), out.stride(0),
        _ptr(lse), batch, heads, len_q, len_k, head_dim, _stream_ptr()), "attention_decode_tc")
    return out, lse


def sample_tokens(logits: torch.Tensor, *, temperature: float, top_p: float, seed: torch.Tensor, step: int,
                  out: torch.Tensor | None = None) -> torch.Tensor:
    """One token per row of logits [rows, V] (fp32 or bf16, unit inner stride, any row pitch): NaN / Inf guards,
    z = logits / temperature, the top-p nucleus (tokens whose strictly-larger-z mass is < top_p), then the
    Gumbel-max draw keyed by Philox4x32-10 of (seed, row, step); the rule is stated in b200_bridge.h.
    `seed` is a one-element int64 CUDA tensor read when the kernel runs. Returns `out` (int64 [rows], any
    stride; allocated when None)."""
    _need_cuda(logits, seed, out)
    if logits.dim() != 2 or logits.stride(1) != 1:
        raise RuntimeError("sample_tokens: logits must be 2-D with unit inner stride")
    if logits.dtype not in (torch.float32, torch.bfloat16):
        raise RuntimeError("sample_tokens: logits must be fp32 or bf16")
    if seed.dtype != torch.int64 or seed.numel() != 1:
        raise RuntimeError("sample_tokens: seed must be a one-element int64 tensor")
    rows, vocab = logits.shape
    if out is None:
        out = torch.empty(rows, device=logits.device, dtype=torch.int64)
    if out.dtype != torch.int64 or out.dim() != 1 or out.shape[0] != rows:
        raise RuntimeError("sample_tokens: `out` must be int64 [rows]")
    ld = logits.stride(0) if rows > 1 else max(logits.stride(0), vocab)
    _lib.check(_lib.lib().b200b_sample_tokens(logits.data_ptr(), 1 if logits.dtype == torch.bfloat16 else 0, ld, rows,
                                              vocab, float(temperature), float(top_p), seed.data_ptr(), int(step),
                                              out.data_ptr(), out.stride(0), _stream_ptr()), "sample_tokens")
    return out


def gemm_grad_pair(dy: torch.Tensor, w: torch.Tensor, x: torch.Tensor, *, wgrad_dtype: torch.dtype = torch.float32):
    """dX = dY W (bf16 [rows, n_in]) and dW = dY^T X ([n_out, n_in], fp32 or bf16) of one Linear through
    b200b_gemm_dual: ONE grouped persistent launch when both fit 256 x 128 pair tiles, two launches otherwise.
    dy bf16 [rows, n_out], w bf16 [n_out, n_in], x bf16 [rows, n_in] (2-D views, any row pitch)."""
    _need_cuda(dy, w, x)
    rows, n_out = dy.shape
    n_in = w.shape[1]
    dx = torch.empty((rows, n_in), device=dy.device, dtype=torch.bfloat16)
    dw = torch.empty((n_out, n_in), device=dy.device, dtype=wgrad_dtype)
    dg = _lib.GemmArgs(a=dy.data_ptr(), b=w.data_ptr(), a_major=0, b_major=1, m=rows, n=n_in, k=n_out, lda=dy.stride(0),
                       ldb=w.stride(0), epilogue=EPI_BF16_BIAS, block_n=0, out=dx.data_ptr(), ldo=dx.stride(0), aux=None,
                       ldaux=0, bias=None, resid=None, ldr=0, beta=0.0, dropout_p=0.0, seed=0, dropout_stream=0, cta_group=0)
    wg = _lib.GemmArgs(a=dy.data_ptr(), b=x.data_ptr(), a_major=1, b_major=1, m=n_out, n=n_in, k=rows, lda=dy.stride(0),
                       ldb=x.stride(0), epilogue=EPI_F32 if wgrad_dtype == torch.float32 else EPI_BF16_BIAS, block_n=0,
                       out=dw.data_ptr(), ldo=dw.stride(0), aux=None, ldaux=0, bias=None, resid=None, ldr=0, beta=0.0,
                       dropout_p=0.0, seed=0, dropout_stream=0, cta_group=0)
    _lib.check(_lib.lib().b200b_gemm_dual(C.byref(dg), C.byref(wg), _stream_ptr()), "gemm_dual")
    return dx, dw
