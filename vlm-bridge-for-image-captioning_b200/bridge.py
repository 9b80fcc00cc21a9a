"""Drop-in `BridgeLite` whose forward/backward run on the sm_100a kernels of libb200_bridge.so.

Mirrors the reference module surface (src/vlm_bridge/model_architecture/bridge_module.py):
  * constructor `(vision_dim, language_dim, num_blocks, num_heads_cross, num_heads_self, dropout)`
    (:350-358), attributes `vision_dim / language_dim / num_blocks / bridge_blocks` (:372-389);
  * `forward(vision_features, text_embeddings, debug=False)` (:406-456) and `get_model_info()`
    (:458-471);
  * the 52-tensor `state_dict` layout and parameter registration order (SURVEY.md Appendix A),
    Xavier-uniform / zero-bias / unit-LayerNorm init consuming the torch RNG exactly like the
    reference (:394-404), so `torch.manual_seed(s); BridgeLite()` yields identical weights.

What differs is only *how* the arithmetic runs: parameters live in one flat fp32 buffer (each
`nn.Parameter` is a view of it), a bf16 copy of the weight region is refreshed when a parameter
version changes, and one `torch.autograd.Function` enqueues whole-block CUDA entry points. Math is
bf16-operand / fp32-accumulate with an fp32 residual stream, i.e. the reference's numerics under
`torch.autocast(dtype=bfloat16)` (SURVEY.md Appendix B), whether or not autocast is active.
There is no CPU or eager-PyTorch fallback: CPU tensors raise.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Optional

import torch
import torch.nn as nn

from . import _lib

__all__ = ["BridgeLite", "BridgeBlock", "MultiHeadCrossAttention", "MultiHeadSelfAttention"]


# ------------------------------------------------------------------------------------------------
# parameter containers: same attribute names / construction order as the reference classes so the
# state_dict keys, registration order and RNG consumption at init are identical
# ------------------------------------------------------------------------------------------------
class MultiHeadCrossAttention(nn.Module):
    """Parameter container of the cross-attention (reference bridge_module.py:24-73)."""

    def __init__(self, query_dim: int, kv_dim: int, d_model: int, num_heads: int = 8, dropout: float = 0.2):
        super().__init__()
        assert d_model % num_heads == 0
        self.query_dim, self.kv_dim, self.d_model, self.num_heads = query_dim, kv_dim, d_model, num_heads
        self.d_k = d_model // num_heads
        self.w_q = nn.Linear(query_dim, d_model)
        self.w_k = nn.Linear(kv_dim, d_model)
        self.w_v = nn.Linear(kv_dim, d_model)
        self.w_o = nn.Linear(d_model, query_dim)
        self.dropout = nn.Dropout(dropout)

    def forward(self, query: torch.Tensor, key: torch.Tensor, value: torch.Tensor, mask=None) -> torch.Tensor:
        """W_o * SDPA(W_q query, W_k key, W_v value) (reference bridge_module.py:75-120), inference only, on the
        library's kernels (tcgen05 GEMMs + fused attention); output bf16-rounded values in fp32 like autocast."""
        _layer_guard("MultiHeadCrossAttention", query, key, value, mask=mask)
        B, Lq, _ = query.shape
        Lk = key.shape[1]
        q = _project(_rows_bf16(query), self.w_q)
        k16 = _rows_bf16(key)
        k = _project(k16, self.w_k)
        v = _project(k16 if value is key else _rows_bf16(value), self.w_v)
        o = _attend(q, k, v, B, Lq, Lk, self.num_heads, self.d_k)
        return _project(o, self.w_o).float().view(B, Lq, self.query_dim)


class MultiHeadSelfAttention(nn.Module):
    """Parameter container of the self-attention (reference bridge_module.py:142-176)."""

    def __init__(self, d_model: int, num_heads: int = 18, dropout: float = 0.2):
        super().__init__()
        assert d_model % num_heads == 0
        self.d_model, self.num_heads = d_model, num_heads
        self.d_k = d_model // num_heads
        self.w_q = nn.Linear(d_model, d_model)
        self.w_k = nn.Linear(d_model, d_model)
        self.w_v = nn.Linear(d_model, d_model)
        self.w_o = nn.Linear(d_model, d_model)
        self.dropout = nn.Dropout(dropout)

    def forward(self, x: torch.Tensor, mask=None) -> torch.Tensor:
        """Non-causal, unmasked self-attention (reference bridge_module.py:178-222), inference only."""
        _layer_guard("MultiHeadSelfAttention", x, mask=mask)
        B, L, _ = x.shape
        x16 = _rows_bf16(x)
        q, k, v = _project(x16, self.w_q), _project(x16, self.w_k), _project(x16, self.w_v)
        o = _attend(q, k, v, B, L, L, self.num_heads, self.d_k)
        return _project(o, self.w_o).float().view(B, L, self.d_model)


class BridgeBlock(nn.Module):
    """Parameter container of one block (reference bridge_module.py:240-298)."""

    def __init__(self, vision_dim: int = 1024, language_dim: int = 2304, num_heads_cross: int = 8,
                 num_heads_self: int = 18, dropout: float = 0.2):
        super().__init__()
        self.vision_dim, self.language_dim = vision_dim, language_dim
        self.cross_attention = MultiHeadCrossAttention(query_dim=language_dim, kv_dim=vision_dim,
                                                       d_model=language_dim, num_heads=num_heads_cross,
                                                       dropout=dropout)
        self.ln_cross = nn.LayerNorm(language_dim)
        self.self_attention = MultiHeadSelfAttention(d_model=language_dim, num_heads=num_heads_self,
                                                     dropout=dropout)
        self.ln_self = nn.LayerNorm(language_dim)
        self.ffn = nn.Sequential(
            nn.Linear(language_dim, language_dim * 4),
            nn.GELU(),
            nn.Dropout(dropout),
            nn.Linear(language_dim * 4, language_dim),
            nn.Dropout(dropout),
        )
        self.ln_ffn = nn.LayerNorm(language_dim)

    def forward(self, text_embeddings: torch.Tensor, vision_features: torch.Tensor) -> torch.Tensor:
        """One block on its own (reference bridge_module.py:300-335), inference only: the three pre-LN residual
        sub-layers through the library's LayerNorm, GEMM (GELU / residual epilogues) and attention kernels."""
        from . import ops
        _layer_guard("BridgeBlock", text_embeddings, vision_features)
        B, L, D = text_embeddings.shape
        x = text_embeddings.detach().to(torch.float32).reshape(B * L, D).contiguous()

        def ln(t, m):
            return ops.layernorm_fwd(t, m.weight.detach().float().contiguous(), m.bias.detach().float().contiguous())[0]

        def out_proj(a16, linear, resid):
            return ops.gemm(a16, _w16(linear), epilogue=ops.EPI_F32_BIAS_RESID, bias=linear.bias.detach().float().contiguous(),
                            resid=resid)

        ca, sa = self.cross_attention, self.self_attention
        v16 = _rows_bf16(vision_features)
        Nv = vision_features.shape[1]
        q = _project(ln(x, self.ln_cross), ca.w_q)
        o = _attend(q, _project(v16, ca.w_k), _project(v16, ca.w_v), B, L, Nv, ca.num_heads, ca.d_k)
        x = out_proj(o, ca.w_o, x)
        xn = ln(x, self.ln_self)
        o = _attend(_project(xn, sa.w_q), _project(xn, sa.w_k), _project(xn, sa.w_v), B, L, L, sa.num_heads, sa.d_k)
        x = out_proj(o, sa.w_o, x)
        h, _u = ops.gemm(ln(x, self.ln_ffn), _w16(self.ffn[0]), epilogue=ops.EPI_BF16_BIAS_GELU,
                         bias=self.ffn[0].bias.detach().float().contiguous())
        x = out_proj(h, self.ffn[3], x)
        return x.view(B, L, D)


# ------------------------------------------------------------------------------------------------
# flat parameter layout
# ------------------------------------------------------------------------------------------------
class _Layout:
    """Element offsets of every parameter inside the flat fp32 buffer.

    Region W (2-D weights, mirrored 1:1 into the bf16 arena):
        [ (w_k, w_v) of block 0, block 1, ... ]                      -> one [nb*2D, Dv] matrix
        per block: cross w_q | cross w_o | self w_q,w_k,w_v ([3D,D]) | self w_o | ffn.0 | ffn.3
    Region V (vectors, fp32 only):
        [ (b_k, b_v) of block 0, block 1, ... ]                      -> one [nb*2D] vector
        per block: cross b_q | cross b_o | self b_q,b_k,b_v ([3D]) | self b_o | ffn.0.b | ffn.3.b |
                   ln_cross w,b | ln_self w,b | ln_ffn w,b
    The gradient arena uses the same offsets, so a block's gradients are two contiguous slabs
    (its W slab and its V slab) -- the data-parallel buckets.
    """

    def __init__(self, nb: int, D: int, Dv: int, F: int):
        self.nb, self.D, self.Dv, self.F = nb, D, Dv, F
        self.offsets: dict[str, int] = {}
        off = 0

        def put(name: str, n: int) -> None:
            nonlocal off
            self.offsets[name] = off
            off += n

        self.kv_w_start = off
        for i in range(nb):
            put(f"bridge_blocks.{i}.cross_attention.w_k.weight", D * Dv)
            put(f"bridge_blocks.{i}.cross_attention.w_v.weight", D * Dv)
        self.block_w_start, self.block_w_end = [], []
        for i in range(nb):
            self.block_w_start.append(off)
            pre = f"bridge_blocks.{i}."
            put(pre + "cross_attention.w_q.weight", D * D)
            put(pre + "cross_attention.w_o.weight", D * D)
            put(pre + "self_attention.w_q.weight", D * D)
            put(pre + "self_attention.w_k.weight", D * D)
            put(pre + "self_attention.w_v.weight", D * D)
            put(pre + "self_attention.w_o.weight", D * D)
            put(pre + "ffn.0.weight", F * D)
            put(pre + "ffn.3.weight", D * F)
            self.block_w_end.append(off)
        self.n_weights = off
        self.kv_b_start = off
        for i in range(nb):
            put(f"bridge_blocks.{i}.cross_attention.w_k.bias", D)
            put(f"bridge_blocks.{i}.cross_attention.w_v.bias", D)
        self.block_v_start, self.block_v_end = [], []
        for i in range(nb):
            self.block_v_start.append(off)
            pre = f"bridge_blocks.{i}."
            put(pre + "cross_attention.w_q.bias", D)
            put(pre + "cross_attention.w_o.bias", D)
            put(pre + "self_attention.w_q.bias", D)
            put(pre + "self_attention.w_k.bias", D)
            put(pre + "self_attention.w_v.bias", D)
            put(pre + "self_attention.w_o.bias", D)
            put(pre + "ffn.0.bias", F)
            put(pre + "ffn.3.bias", D)
            for ln in ("ln_cross", "ln_self", "ln_ffn"):
                put(pre + ln + ".weight", D)
                put(pre + ln + ".bias", D)
            self.block_v_end.append(off)
        self.total = off

    def buckets(self) -> list[tuple[int, int]]:
        """(start, end) element ranges in the order backward finishes them (last block first)."""
        out = []
        for i in reversed(range(self.nb)):
            out.append((self.block_w_start[i], self.block_w_end[i]))
            out.append((self.block_v_start[i], self.block_v_end[i]))
        out.append((self.kv_w_start, self.block_w_start[0]))
        out.append((self.kv_b_start, self.block_v_start[0]))
        return out


# ------------------------------------------------------------------------------------------------
# per-layer forwards (inference only): the reference exports these classes as working modules
# (model_architecture/__init__.py:22-27). Training goes through BridgeLite's fused autograd node; the
# layers on their own run the same kernels through the thin op wrappers, without autograd.
# ------------------------------------------------------------------------------------------------
def _layer_guard(name: str, *tensors: torch.Tensor, mask=None) -> None:
    if mask is not None:
        raise RuntimeError(f"{name}: attention masks are not built (the bridge never passes one: "
                           "bridge_module.py:317-322,327)")
    for t in tensors:
        if not t.is_cuda:
            raise RuntimeError(f"{name} (B200) runs on CUDA only: there is no CPU fallback")
    if torch.is_grad_enabled() and any(t.requires_grad for t in tensors):
        raise RuntimeError(f"{name}.forward on its own is inference-only (wrap it in torch.no_grad()); training runs "
                           "through BridgeLite.forward, which fuses the layers into one autograd node")


def _w16(linear: nn.Linear) -> torch.Tensor:
    return linear.weight.detach().to(torch.bfloat16).contiguous()


def _rows_bf16(x: torch.Tensor) -> torch.Tensor:
    from . import ops
    x2 = x.detach().reshape(-1, x.shape[-1])
    return x2.contiguous() if x2.dtype == torch.bfloat16 else ops.cast_bf16(x2.to(torch.float32).contiguous())


def _project(x16: torch.Tensor, linear: nn.Linear) -> torch.Tensor:
    from . import ops
    return ops.gemm(x16, _w16(linear), bias=linear.bias.detach().float().contiguous())


def _attend(q16, k16, v16, batch, len_q, len_k, heads, d_k) -> torch.Tensor:
    from . import ops
    if d_k not in (64, 128, 288):
        raise RuntimeError(f"attention kernels are built for head dims 64 / 128 / 288, not {d_k}")
    o, _ = ops.attention_fwd(q16, k16, v16, batch=batch, heads=heads, len_q=len_q, len_k=len_k, head_dim=d_k)
    return o


class _BridgeDims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("batch", "len_text", "len_vision", "dim", "dim_vision", "dim_ffn",
                                         "heads_cross", "heads_self", "num_blocks", "flags")]


FLAG_WGRAD_BF16 = 1      # B200B_BRIDGE_WGRAD_BF16
FLAG_SEED_INDIRECT = 2   # B200B_BRIDGE_SEED_INDIRECT
FLAG_KV_PACKED = 4       # B200B_BRIDGE_KV_PACKED
FLAG_KV_TC = 8           # B200B_BRIDGE_KV_TC
FLAG_PART_CROSS = 16     # B200B_BRIDGE_PART_CROSS
FLAG_PART_REST = 32      # B200B_BRIDGE_PART_REST
TC_DECODE_MIN_LEN = 33   # prefix lengths from which the tcgen05 decode kernel beats the mma.sync one (measured)
_SEED_STRIDE = 0x1E3779B97F4A7C15  # odd 61-bit increment of the device-resident dropout seed
_GRAD_READY_FN = C.CFUNCTYPE(None, C.c_void_p, C.c_void_p, C.c_int64)


class _GradNotify(C.Structure):
    _fields_ = [("fn", _GRAD_READY_FN), ("user", C.c_void_p)]


_W_FIELDS = ["wq_c", "wo_c", "wqkv_s", "wo_s", "w1", "w2", "bq_c", "bo_c", "bqkv_s", "bo_s", "b1", "b2",
             "ln_c_g", "ln_c_b", "ln_s_g", "ln_s_b", "ln_f_g", "ln_f_b"]
_W_KEYS = ["cross_attention.w_q.weight", "cross_attention.w_o.weight", "self_attention.w_q.weight",
           "self_attention.w_o.weight", "ffn.0.weight", "ffn.3.weight", "cross_attention.w_q.bias",
           "cross_attention.w_o.bias", "self_attention.w_q.bias", "self_attention.w_o.bias", "ffn.0.bias",
           "ffn.3.bias", "ln_cross.weight", "ln_cross.bias", "ln_self.weight", "ln_self.bias", "ln_ffn.weight",
           "ln_ffn.bias"]


class _BlockPtrs(C.Structure):
    """b200b_block_weights and b200b_block_grads share this shape (18 pointers)."""
    _fields_ = [(n, C.c_void_p) for n in _W_FIELDS]


def _declare_bridge(lib) -> None:
    if getattr(lib, "_b200b_bridge_declared", False):
        return
    P = C.POINTER
    lib.b200b_bridge_block_saved_bytes.restype = C.c_size_t
    lib.b200b_bridge_block_saved_bytes.argtypes = [P(_BridgeDims)]
    lib.b200b_bridge_backward_workspace_bytes.restype = C.c_size_t
    lib.b200b_bridge_backward_workspace_bytes.argtypes = [P(_BridgeDims)]
    lib.b200b_bridge_kv_project.restype = C.c_int
    lib.b200b_bridge_kv_project.argtypes = [P(_BridgeDims)] + [C.c_void_p] * 6
    lib.b200b_bridge_block_forward.restype = C.c_int
    lib.b200b_bridge_block_forward.argtypes = [P(_BridgeDims), C.c_int, P(_BlockPtrs), C.c_void_p, C.c_void_p,
                                               C.c_void_p, C.c_void_p, C.c_size_t, C.c_float, C.c_uint64,
                                               C.c_void_p]
    lib.b200b_bridge_block_backward.restype = C.c_int
    lib.b200b_bridge_block_backward.argtypes = [P(_BridgeDims), C.c_int, P(_BlockPtrs), C.c_void_p, C.c_void_p,
                                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, P(_BlockPtrs),
                                                C.c_void_p, C.c_size_t, C.c_float, C.c_uint64, P(_GradNotify),
                                                C.c_void_p]
    lib.b200b_bridge_kv_backward.restype = C.c_int
    lib.b200b_bridge_kv_backward.argtypes = [P(_BridgeDims), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_size_t, C.c_void_p]
    lib.b200b_bridge_f32_workspace_bytes.restype = C.c_size_t
    lib.b200b_bridge_f32_workspace_bytes.argtypes = [P(_BridgeDims)]
    lib.b200b_bridge_kv_project_f32.restype = C.c_int
    lib.b200b_bridge_kv_project_f32.argtypes = [P(_BridgeDims)] + [C.c_void_p] * 5
    lib.b200b_bridge_block_forward_f32.restype = C.c_int
    lib.b200b_bridge_block_forward_f32.argtypes = [P(_BridgeDims), C.c_int, P(_BlockPtrs), C.c_void_p, C.c_void_p,
                                                   C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib._b200b_bridge_declared = True


def _bridge_lib():
    lib = _lib.lib()
    _declare_bridge(lib)
    return lib


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# ------------------------------------------------------------------------------------------------
# the autograd function: one node for the whole bridge
# ------------------------------------------------------------------------------------------------
class _BridgeFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, module: "BridgeLite", vision: torch.Tensor, text: torch.Tensor, *params: torch.Tensor):
        out, state = module._run_forward(vision, text, keep_for_backward=True)
        ctx.module = module
        ctx.state = state
        ctx.text_needs_grad = text.requires_grad
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, d_out: torch.Tensor):
        module: BridgeLite = ctx.module
        # the saved activations stay with ctx (freed with the graph), so backward(retain_graph=True) works
        d_text, grads = module._run_backward(ctx.state, d_out, ctx.text_needs_grad)
        return (None, None, d_text, *grads)


class BridgeLite(nn.Module):
    """Bridge-Lite on B200: same constructor, forward signature and state_dict as the reference
    `BridgeLite` (bridge_module.py:338-471)."""

    def __init__(self, vision_dim: int = 1024, language_dim: int = 2304, num_blocks: int = 2,
                 num_heads_cross: int = 8, num_heads_self: int = 18, dropout: float = 0.2):
        super().__init__()
        self.vision_dim = vision_dim
        self.language_dim = language_dim
        self.num_blocks = num_blocks
        self.num_heads_cross = num_heads_cross
        self.num_heads_self = num_heads_self
        self.dropout_p = float(dropout)
        self.bridge_blocks = nn.ModuleList([
            BridgeBlock(vision_dim=vision_dim, language_dim=language_dim, num_heads_cross=num_heads_cross,
                        num_heads_self=num_heads_self, dropout=dropout) for _ in range(num_blocks)
        ])
        self._init_weights()
        self._layout = _Layout(num_blocks, language_dim, vision_dim, language_dim * 4)
        # lazily built device state (never part of state_dict)
        self._flat: Optional[torch.Tensor] = None
        self._w16: Optional[torch.Tensor] = None
        self._w16_key = None
        self._ptrs = None
        # data-parallel reducer (parallel.GradBucketReducer) driven by _run_backward
        self._bucket_hook = None
        self._last_grad_arena: Optional[torch.Tensor] = None
        self._grad16: Optional[torch.Tensor] = None      # averaged bf16 weight gradients not yet materialised as .grad
        self._graph_recast = True

    # -- init exactly as the reference (bridge_module.py:394-404) ---------------------------------
    def _init_weights(self) -> None:
        for module in self.modules():
            if isinstance(module, nn.Linear):
                nn.init.xavier_uniform_(module.weight)
                if module.bias is not None:
                    nn.init.zeros_(module.bias)
            elif isinstance(module, nn.LayerNorm):
                nn.init.ones_(module.weight)
                nn.init.zeros_(module.bias)

    # -- flat parameter storage --------------------------------------------------------------------
    def _named_params(self) -> list[tuple[str, nn.Parameter]]:
        """(name, parameter) in registration order. Walking the module tree costs ~0.1 ms and a step
        needs the list several times, so it is cached; the cache is checked against the owning
        modules' `_parameters` dicts (one identity test per tensor), which catches a parameter that
        was re-assigned, and dropped by `_apply` (.to / .cuda / .float)."""
        cache = self.__dict__.get("_plist_cache")
        if cache is not None:
            for owner, key, _name, p in cache:
                if owner._parameters.get(key) is not p:
                    cache = None
                    break
        if cache is None:
            cache = []
            for mod_name, mod in self.named_modules():
                for key, p in mod._parameters.items():
                    if p is not None:
                        cache.append((mod, key, (mod_name + "." if mod_name else "") + key, p))
            self.__dict__["_plist_cache"] = cache
        return [(name, p) for _, _, name, p in cache]

    def _apply(self, fn, *args, **kwargs):
        self.__dict__["_plist_cache"] = None
        return super()._apply(fn, *args, **kwargs)

    def _ensure_flat(self) -> None:
        """Make every parameter a view of one flat fp32 CUDA buffer (re-done after .to()/.cuda())."""
        named = self._named_params()
        dev = named[0][1].device
        if dev.type != "cuda":
            raise RuntimeError("BridgeLite (B200) runs on CUDA only: move the module to a cuda device "
                               "(there is no CPU fallback)")
        lay = self._layout
        flat = self._flat
        ok = flat is not None and flat.device == dev
        if ok:
            base = flat.data_ptr()
            for name, p in named:
                if p.dtype != torch.float32 or p.data_ptr() != base + 4 * lay.offsets[name]:
                    ok = False
                    break
        if ok:
            return
        for _, p in named:
            if p.dtype != torch.float32:
                raise RuntimeError("BridgeLite (B200) keeps fp32 master parameters; do not cast the module "
                                   "to half precision (bf16 operand copies are made internally)")
        flat = torch.empty(lay.total, device=dev, dtype=torch.float32)
        with torch.no_grad():
            for name, p in named:
                o = lay.offsets[name]
                view = flat[o:o + p.numel()].view(p.shape)
                view.copy_(p.data)
                p.data = view
        self._flat = flat
        # device-resident dropout seed, used (and advanced by a captured kernel) under CUDA-graph capture
        self._seed_dev = torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).to(dev)
        self._w16 = torch.empty(lay.n_weights, device=dev, dtype=torch.bfloat16)
        self._w16_key = None
        self._ptrs = None

    def _refresh_bf16(self) -> None:
        key = tuple(p._version for _, p in self._named_params())
        # while a CUDA graph is being captured the cast is always recorded: the optimizer updates the
        # fp32 masters between replays without this code running again (inference graphs, whose weights
        # are frozen for the graph's lifetime, opt out through `_graph_recast`)
        if key == self._w16_key and not (torch.cuda.is_current_stream_capturing() and self._graph_recast):
            return
        lay = self._layout
        _lib.check(_lib.lib().b200b_cast_bf16(self._flat.data_ptr(), self._w16.data_ptr(), lay.n_weights, 0.0, 0, 0,
                                              _stream()), "cast_bf16(weights)")
        self._w16_key = key

    def _block_ptr_struct(self, base16: int, base32: int, i: int, grads: bool, esize16: int = 2) -> _BlockPtrs:
        """Pointers of block i's tensors: 2-D weights at base16 (a separate weight arena of
        `esize16`-byte elements) when base16 is given, everything else at base32 (fp32 arena), both at
        the flat-layout offsets."""
        lay = self._layout
        s = _BlockPtrs()
        pre = f"bridge_blocks.{i}."
        for field, key in zip(_W_FIELDS, _W_KEYS):
            off = lay.offsets[pre + key]
            if off < lay.n_weights and base16:
                setattr(s, field, base16 + esize16 * off)
            else:
                setattr(s, field, base32 + 4 * off)
        return s

    def _weight_ptrs(self):
        if self._ptrs is None:
            b16, b32 = self._w16.data_ptr(), self._flat.data_ptr()
            self._ptrs = [self._block_ptr_struct(b16, b32, i, grads=False) for i in range(self.num_blocks)]
        return self._ptrs

    def _dims(self, B: int, L: int, Nv: int, flags: int = 0) -> _BridgeDims:
        return _BridgeDims(batch=B, len_text=L, len_vision=Nv, dim=self.language_dim, dim_vision=self.vision_dim,
                           dim_ffn=self.language_dim * 4, heads_cross=self.num_heads_cross,
                           heads_self=self.num_heads_self, num_blocks=self.num_blocks, flags=flags)

    # -- vision K/V (shared with the decode cache) -------------------------------------------------
    def project_vision_kv(self, vision_features: torch.Tensor, out=None, _weights_current: bool = False):
        """K/V of every block for `vision_features` [B, Nv, vision_dim] -> (vision_bf16, kv bf16
        [B*Nv, num_blocks*2*language_dim]). Reference: bridge_module.py:99-100. `out=(vision_bf16, kv)`
        writes into existing tensors of those shapes."""
        if not _weights_current:        # _run_forward has just refreshed them (under graph capture a second call
            self._ensure_flat()         # would record a second 158 M-element cast into the graph)
            self._refresh_bf16()
        v = vision_features.detach().to(device=self._flat.device, dtype=torch.float32).contiguous()
        B, Nv, Dv = v.shape
        if Dv != self.vision_dim:
            raise RuntimeError(f"vision_features last dim {Dv} != vision_dim {self.vision_dim}")
        lay = self._layout
        D = self.language_dim
        if out is not None:
            vb, kv = out
            if tuple(vb.shape) != (B * Nv, Dv) or tuple(kv.shape) != (B * Nv, self.num_blocks * 2 * D):
                raise RuntimeError("project_vision_kv: out tensors have the wrong shape")
        else:
            vb = torch.empty((B * Nv, Dv), device=v.device, dtype=torch.bfloat16)
            kv = torch.empty((B * Nv, self.num_blocks * 2 * D), device=v.device, dtype=torch.bfloat16)
        dims = self._dims(B, 1, Nv)
        _lib.check(_bridge_lib().b200b_bridge_kv_project(
            C.byref(dims), v.data_ptr(), self._w16.data_ptr() + 2 * lay.kv_w_start,
            self._flat.data_ptr() + 4 * lay.kv_b_start, vb.data_ptr(), kv.data_ptr(), _stream()), "kv_project")
        return vb, kv

    def project_vision_kv_fp32(self, vision_features: torch.Tensor) -> torch.Tensor:
        """fp32 K/V of every block, [B*Nv, num_blocks*2*language_dim], from the fp32 master weights: the
        decode numerics of the reference, which runs generate_caption without autocast
        (full_model.py:221-261 -> bridge_module.py:99-100)."""
        self._ensure_flat()
        v = vision_features.detach().to(device=self._flat.device, dtype=torch.float32).contiguous()
        B, Nv, Dv = v.shape
        if Dv != self.vision_dim:
            raise RuntimeError(f"vision_features last dim {Dv} != vision_dim {self.vision_dim}")
        lay = self._layout
        kv = torch.empty((B * Nv, self.num_blocks * 2 * self.language_dim), device=v.device, dtype=torch.float32)
        dims = self._dims(B, 1, Nv)
        _lib.check(_bridge_lib().b200b_bridge_kv_project_f32(
            C.byref(dims), v.data_ptr(), self._flat.data_ptr() + 4 * lay.kv_w_start,
            self._flat.data_ptr() + 4 * lay.kv_b_start, kv.data_ptr(), _stream()), "kv_project_f32")
        return kv

    def pack_vision_kv(self, kv: torch.Tensor, batch: int, len_vision: int, out=None) -> torch.Tensor:
        """Decode layout of a `project_vision_kv` result: [B][blocks][heads][2][Nv][d+8] bf16 (flat uint8)."""
        lib = _bridge_lib()
        d = self.language_dim // self.num_heads_cross
        nbytes = lib.b200b_kv_cache_packed_bytes(batch, len_vision, self.num_heads_cross, d, self.num_blocks)
        packed = torch.empty(nbytes, device=kv.device, dtype=torch.uint8) if out is None else out
        if packed.numel() != nbytes:
            raise RuntimeError("pack_vision_kv: out has the wrong size")
        _lib.check(lib.b200b_kv_cache_pack(kv.data_ptr(), kv.stride(0), packed.data_ptr(), batch, len_vision,
                                           self.num_heads_cross, d, self.num_blocks, _stream()), "kv_cache_pack")
        return packed

    def pack_vision_kv_tc(self, kv: torch.Tensor, batch: int, len_vision: int, out=None) -> torch.Tensor:
        """tcgen05 decode layout of a `project_vision_kv` result (csrc/attention_tc.cu): per image / block /
        head, 32-key tiles stored as the swizzled shared-memory images the MMAs read."""
        lib = _bridge_lib()
        d = self.language_dim // self.num_heads_cross
        nbytes = lib.b200b_kv_cache_tc_bytes(batch, len_vision, self.num_heads_cross, d, self.num_blocks)
        packed = torch.empty(nbytes, device=kv.device, dtype=torch.uint8) if out is None else out
        if packed.numel() != nbytes:
            raise RuntimeError("pack_vision_kv_tc: out has the wrong size")
        _lib.check(lib.b200b_kv_cache_pack_tc(kv.data_ptr(), kv.stride(0), packed.data_ptr(), batch, len_vision,
                                              self.num_heads_cross, d, self.num_blocks, _stream()), "kv_cache_pack_tc")
        return packed

    # -- forward / backward drivers ----------------------------------------------------------------
    def _kv_flag(self, kv_cache, L: int, keep_for_backward: bool):
        """(kv tensor, B200B_BRIDGE_KV_* flag) a cross-attention over L text positions reads from `kv_cache`."""
        packed = (kv_cache is not None and not keep_for_backward and L <= 64 and not (self.training and self.dropout_p > 0)
                  and getattr(kv_cache, "kv_packed", None) is not None
                  and (self.language_dim // self.num_heads_cross) in (64, 128, 288))
        if not packed:
            return kv_cache.kv, 0
        if L >= TC_DECODE_MIN_LEN and getattr(kv_cache, "kv_tc", None) is not None:
            return kv_cache.kv_tc, FLAG_KV_TC
        return kv_cache.kv_packed, FLAG_KV_PACKED

    def _run_forward(self, vision: torch.Tensor, text: torch.Tensor, keep_for_backward: bool, kv_cache=None,
                     block_callback=None, cached_positions: Optional[int] = None):
        if kv_cache is not None and getattr(kv_cache, "beams", 1) > 1:
            if keep_for_backward:
                raise RuntimeError("a beam-search cache is inference-only")
            return self._run_forward_beams(text, kv_cache, block_callback, cached_positions), None
        self._ensure_flat()
        self._refresh_bf16()
        dev = self._flat.device
        if text.device != dev:
            raise RuntimeError("text_embeddings must be on the module's CUDA device")
        if text.dim() != 3 or text.shape[-1] != self.language_dim:
            raise RuntimeError(f"text_embeddings must be [B, L, {self.language_dim}]")
        x = text.detach().to(torch.float32).contiguous()
        B, L, D = x.shape
        if kv_cache is None:
            if vision.dim() != 3 or vision.shape[0] != B:
                raise RuntimeError("vision_features must be [B, Nv, vision_dim] with the text batch size")
            vb, kv = self.project_vision_kv(vision, _weights_current=True)
            Nv = vision.shape[1]
        else:
            vb, kv, Nv = None, kv_cache.kv, kv_cache.len_vision
            if kv_cache.batch != B:
                raise RuntimeError("kv cache batch does not match text batch")
        lib = _bridge_lib()
        dims = self._dims(B, L, Nv)
        kv_flag = 0
        if kv_cache is not None:
            kv, kv_flag = self._kv_flag(kv_cache, L, keep_for_backward)
        saved_bytes = lib.b200b_bridge_block_saved_bytes(C.byref(dims))
        n_arenas = self.num_blocks if keep_for_backward else 1
        saved = torch.empty(n_arenas * saved_bytes, device=dev, dtype=torch.uint8)
        p = self.dropout_p if self.training else 0.0
        seed, flags = 0, 0
        if p > 0:
            if torch.cuda.is_current_stream_capturing():
                # a host-drawn seed would be baked into the graph: keep it in device memory, advance it
                # with a captured kernel, and let every dropout kernel read it when it runs
                self._seed_dev.add_(_SEED_STRIDE)
                seed, flags = self._seed_dev.data_ptr(), FLAG_SEED_INDIRECT
            else:
                seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        dims = self._dims(B, L, Nv, flags | kv_flag)
        ptrs = self._weight_ptrs()
        xs = [x.view(B * L, D)]
        st = _stream()
        # decode: block 0's cross-attention sub-layer is row-wise in the text (a row of its output depends
        # on the same text row and on the image only), so its rows are kept per position in the cache and
        # only the rows from `cached_positions` on are computed (SURVEY.md 8f rank 2)
        pos_cache = None
        if cached_positions is not None:
            if kv_cache is None or keep_for_backward or p > 0:
                raise RuntimeError("cached_positions needs kv_cache, inference mode and no active dropout")
            pos_cache = kv_cache.position_rows(L, cached_positions, dev, D)
        for i in range(self.num_blocks):
            x_out = torch.empty((B * L, D), device=dev, dtype=torch.float32)
            arena = saved.data_ptr() + (i if keep_for_backward else 0) * saved_bytes
            x_in, bdims = xs[-1], dims
            if i == 0 and pos_cache is not None:
                k = int(cached_positions)
                n_new = L - k
                x_new = x[:, k:, :].contiguous()
                kv_c, flag_c = self._kv_flag(kv_cache, n_new, False)
                cdims = self._dims(B, n_new, Nv, flag_c | FLAG_PART_CROSS)
                x1_new = torch.empty((B * n_new, D), device=dev, dtype=torch.float32)
                _lib.check(lib.b200b_bridge_block_forward(C.byref(cdims), 0, C.byref(ptrs[0]), x_new.data_ptr(),
                                                          kv_c.data_ptr(), x1_new.data_ptr(), arena, saved_bytes, 0.0, 0,
                                                          st), "block_forward(cross part)")
                pos_cache[:, k:L].copy_(x1_new.view(B, n_new, D))
                x_in = pos_cache[:, :L].contiguous().view(B * L, D)
                bdims = self._dims(B, L, Nv, FLAG_PART_REST)
            _lib.check(lib.b200b_bridge_block_forward(C.byref(bdims), i, C.byref(ptrs[i]), x_in.data_ptr(),
                                                      kv.data_ptr(), x_out.data_ptr(), arena, saved_bytes, p, seed,
                                                      st), "block_forward")
            if block_callback is not None:
                block_callback(i, xs[-1].view(B, L, D), x_out.view(B, L, D))
            xs.append(x_out)
        out = xs[-1].view(B, L, D)
        state = None
        if keep_for_backward:
            state = dict(dims=dims, saved=saved, saved_bytes=saved_bytes, kv=kv, vb=vb, xs=xs[:-1], p=p, seed=seed,
                         flags=flags,
                         versions=self._w16_key)
        return out, state

    def _run_forward_fp32(self, text: torch.Tensor, kv_cache, block_callback=None,
                          cached_positions: Optional[int] = None) -> torch.Tensor:
        """Inference forward with fp32 operands over an fp32 `VisionKVCache` (csrc/exact_fp32.cu): the
        reference's decode numerics (no autocast, full_model.py:221-261). Same block / position-row
        structure as `_run_forward`."""
        if getattr(kv_cache, "beams", 1) > 1:
            return self._run_forward_beams(text, kv_cache, block_callback, cached_positions)
        self._ensure_flat()
        dev = self._flat.device
        if self.training and self.dropout_p > 0:
            raise RuntimeError("the fp32 path is inference-only: call .eval() first")
        if text.device != dev or text.dim() != 3 or text.shape[-1] != self.language_dim:
            raise RuntimeError(f"text_embeddings must be a CUDA tensor [B, L, {self.language_dim}] on the module's device")
        x = text.detach().to(torch.float32).contiguous()
        B, L, D = x.shape
        if kv_cache.batch != B:
            raise RuntimeError("kv cache batch does not match text batch")
        Nv = kv_cache.len_vision
        lib = _bridge_lib()
        dims = self._dims(B, L, Nv)
        ws_bytes = lib.b200b_bridge_f32_workspace_bytes(C.byref(dims))
        ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
        ptrs = self._f32_ptrs()
        st = _stream()
        kv = kv_cache.kv32
        pos_cache = None
        if cached_positions is not None:
            pos_cache = kv_cache.position_rows(L, cached_positions, dev, D)
        cur = x.view(B * L, D)
        for i in range(self.num_blocks):
            x_out = torch.empty((B * L, D), device=dev, dtype=torch.float32)
            x_in, bdims = cur, dims
            if i == 0 and pos_cache is not None:
                k = int(cached_positions)
                n_new = L - k
                x_new = x[:, k:, :].contiguous()
                cdims = self._dims(B, n_new, Nv, FLAG_PART_CROSS)
                x1_new = torch.empty((B * n_new, D), device=dev, dtype=torch.float32)
                _lib.check(lib.b200b_bridge_block_forward_f32(C.byref(cdims), 0, C.byref(ptrs[0]), x_new.data_ptr(),
                                                              kv.data_ptr(), x1_new.data_ptr(), ws.data_ptr(), ws_bytes, st),
                           "block_forward_f32(cross part)")
                pos_cache[:, k:L].copy_(x1_new.view(B, n_new, D))
                x_in = pos_cache[:, :L].contiguous().view(B * L, D)
                bdims = self._dims(B, L, Nv, FLAG_PART_REST)
            _lib.check(lib.b200b_bridge_block_forward_f32(C.byref(bdims), i, C.byref(ptrs[i]), x_in.data_ptr(),
                                                          kv.data_ptr(), x_out.data_ptr(), ws.data_ptr(), ws_bytes, st),
                       "block_forward_f32")
            if block_callback is not None:
                block_callback(i, cur.view(B, L, D), x_out.view(B, L, D))
            cur = x_out
        return cur.view(B, L, D)

    def _f32_ptrs(self):
        """Block pointer structs of the fp32 path (every field in the fp32 arena), cached per arena address."""
        b32 = self._flat.data_ptr()
        ptrs = self.__dict__.get("_ptrs32")
        if ptrs is None or ptrs[0] != b32:
            ptrs = (b32, [self._block_ptr_struct(0, b32, i, grads=False) for i in range(self.num_blocks)])
            self.__dict__["_ptrs32"] = ptrs
        return ptrs[1]

    def _run_forward_beams(self, text: torch.Tensor, kv_cache, block_callback=None,
                           cached_positions: Optional[int] = None) -> torch.Tensor:
        """Inference forward over a beam-search cache (`VisionKVCache(..., beams=K)`, either precision): text
        [B*K, L, D], rows [B][K][L], over the K/V of B images. Every block runs as two calls on the same buffers:
        the cross-attention sub-layer with dims (batch=B, len_text=K*L) -- image b's K*L rows are one query block
        over its cache, which is read once for all its beams -- and the rest of the block with dims
        (batch=B*K, len_text=L), so that the self-attention and the FFN stay within a beam. Both dims come from
        the cache's (batch, beams), after the text batch is checked against them."""
        B, K = int(kv_cache.batch), int(kv_cache.beams)
        if text.dim() != 3 or int(text.shape[0]) != B * K:
            raise RuntimeError(f"a cache of {B} images x {K} beams needs text_embeddings [{B * K}, L, "
                               f"{self.language_dim}], got {tuple(text.shape)}")
        self._ensure_flat()
        fp32 = kv_cache.precision == "fp32"
        if self.training and self.dropout_p > 0:
            raise RuntimeError("a beam-search cache needs inference mode: call .eval() first")
        if not fp32:
            self._refresh_bf16()
        dev = self._flat.device
        if text.device != dev or text.shape[-1] != self.language_dim:
            raise RuntimeError(f"text_embeddings must be a CUDA tensor [B*K, L, {self.language_dim}] on the module's device")
        x = text.detach().to(torch.float32).contiguous()
        _, L, D = x.shape
        Nv = kv_cache.len_vision
        lib = _bridge_lib()
        st = _stream()
        pos_cache, k0 = None, 0
        if cached_positions is not None:
            pos_cache = kv_cache.position_rows(L, cached_positions, dev, D)
            k0 = int(cached_positions) if pos_cache is not None else 0
        rdims = self._dims(B * K, L, Nv, FLAG_PART_REST)
        full_cross = self._dims(B, K * L, Nv, FLAG_PART_CROSS)
        if fp32:
            ptrs, kv = self._f32_ptrs(), kv_cache.kv32
            ws_bytes = max(lib.b200b_bridge_f32_workspace_bytes(C.byref(d)) for d in (rdims, full_cross))
        else:
            ptrs, kv = self._weight_ptrs(), kv_cache.kv
            ws_bytes = max(lib.b200b_bridge_block_saved_bytes(C.byref(d)) for d in (rdims, full_cross))
        ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)

        def block(dims, i, x_in, kv_t, x_out, what):
            if fp32:
                rc = lib.b200b_bridge_block_forward_f32(C.byref(dims), i, C.byref(ptrs[i]), x_in.data_ptr(), kv_t.data_ptr(),
                                                        x_out.data_ptr(), ws.data_ptr(), ws_bytes, st)
            else:
                rc = lib.b200b_bridge_block_forward(C.byref(dims), i, C.byref(ptrs[i]), x_in.data_ptr(), kv_t.data_ptr(),
                                                    x_out.data_ptr(), ws.data_ptr(), ws_bytes, 0.0, 0, st)
            _lib.check(rc, what)

        def cross(i, x_in, n):
            """x1 [B*K*n, D] of the cross-attention sub-layer for n positions of every beam"""
            kv_t, flag = (kv, 0) if fp32 else self._kv_flag(kv_cache, K * n, False)
            x1 = torch.empty((B * K * n, D), device=dev, dtype=torch.float32)
            block(self._dims(B, K * n, Nv, flag | FLAG_PART_CROSS), i, x_in, kv_t, x1, "block_forward(beams, cross part)")
            return x1

        cur = x.view(B * K * L, D)
        for i in range(self.num_blocks):
            if i == 0 and pos_cache is not None:
                n_new = L - k0
                x1_new = cross(0, x[:, k0:, :].contiguous(), n_new)
                pos_cache[:, k0:L].copy_(x1_new.view(B * K, n_new, D))
                x1 = pos_cache[:, :L].contiguous().view(B * K * L, D)
            else:
                x1 = cross(i, cur, L)
            x_out = torch.empty((B * K * L, D), device=dev, dtype=torch.float32)
            block(rdims, i, x1, kv, x_out, "block_forward(beams, rest)")
            if block_callback is not None:
                block_callback(i, cur.view(B * K, L, D), x_out.view(B * K, L, D))
            cur = x_out
        return cur.view(B * K, L, D)

    def _run_backward(self, state, d_out: torch.Tensor, text_needs_grad: bool):
        lay = self._layout
        dev = self._flat.device
        lib = _bridge_lib()
        fdims = state["dims"]
        if state["versions"] != tuple(p._version for _, p in self._named_params()):
            raise RuntimeError("bridge parameters were modified in place between forward and backward")
        B, L, D = fdims.batch, fdims.len_text, fdims.dim
        d = d_out.detach().to(torch.float32).contiguous().view(B * L, D)
        # data parallel: `reducer` exchanges gradient ranges as soon as their kernels are enqueued.
        # With a bf16 exchange the weight-gradient GEMMs write a bf16 arena (the values autocast gives
        # these gradients in the reference) and the averaged buckets end up as fp32 in garena. The nvls
        # transport owns both arenas (symmetric memory, reused every step).
        reducer = self._bucket_hook
        garena = None
        g16 = None   # arena the weight-gradient GEMMs write when it is not garena itself
        if reducer is not None and reducer.world_size > 1:
            garena, g16 = reducer.arenas(lay.n_weights, lay.total, dev)
            if garena is not None:
                # a persistent arena: gradients still referenced from an earlier step (accumulation
                # without zero_grad) must not be overwritten in place
                lo_, hi_ = garena.data_ptr(), garena.data_ptr() + 4 * lay.total
                for _, p_ in self._named_params():
                    if p_.grad is not None and lo_ <= p_.grad.data_ptr() < hi_ and not torch.cuda.is_current_stream_capturing():
                        p_.grad = p_.grad.clone()
            elif reducer.wgrad_bf16:
                g16 = torch.empty(lay.n_weights, device=dev, dtype=torch.bfloat16)
        if garena is None:
            garena = torch.empty(lay.total, device=dev, dtype=torch.float32)
        gbase = garena.data_ptr()
        wgrad_bf16 = g16 is not None and g16.dtype == torch.bfloat16
        g16base = g16.data_ptr() if g16 is not None else 0
        g16size = g16.element_size() if g16 is not None else 4
        dims = self._dims(B, L, fdims.len_vision, (FLAG_WGRAD_BF16 if wgrad_bf16 else 0) | state["flags"])
        ws_bytes = lib.b200b_bridge_backward_workspace_bytes(C.byref(dims))
        ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
        dkv = torch.empty_like(state["kv"])
        ptrs = self._weight_ptrs()
        st = _stream()
        notify = None
        if reducer is not None:
            reducer.begin(garena, g16, lay.n_weights)
            wbase, wsize = (g16base, g16size) if g16 is not None else (gbase, 4)

            cb_errors: list[BaseException] = []

            def _ready(_user, ptr, elems):
                try:                                  # an exception cannot cross the C frame: keep it
                    start = (ptr - wbase) // wsize
                    reducer.weights_ready(start, start + elems)
                except BaseException as e:  # noqa: BLE001
                    cb_errors.append(e)

            cb = _GRAD_READY_FN(_ready)            # kept alive until the end of this function
            notify = _GradNotify(cb, None)
        for i in reversed(range(self.num_blocks)):
            need_din = i > 0 or text_needs_grad
            d_in = torch.empty((B * L, D), device=dev, dtype=torch.float32) if need_din else None
            g = self._block_ptr_struct(g16base, gbase, i, grads=True, esize16=g16size)
            arena = state["saved"].data_ptr() + i * state["saved_bytes"]
            _lib.check(lib.b200b_bridge_block_backward(
                C.byref(dims), i, C.byref(ptrs[i]), state["xs"][i].data_ptr(), state["kv"].data_ptr(), arena,
                d.data_ptr(), None if d_in is None else d_in.data_ptr(), dkv.data_ptr(), C.byref(g), ws.data_ptr(),
                ws_bytes, state["p"], state["seed"], None if notify is None else C.byref(notify), st),
                "block_backward")
            if reducer is not None:
                if cb_errors:
                    raise cb_errors[0]
                reducer.flush()
                reducer.vectors_ready(lay.block_v_start[i], lay.block_v_end[i])
            d = d_in
        _lib.check(lib.b200b_bridge_kv_backward(
            C.byref(dims), state["vb"].data_ptr(), dkv.data_ptr(),
            (g16base + g16size * lay.kv_w_start) if g16 is not None else (gbase + 4 * lay.kv_w_start),
            gbase + 4 * lay.kv_b_start, ws.data_ptr(), ws_bytes, st), "kv_backward")
        if reducer is not None:
            reducer.weights_ready(lay.kv_w_start, lay.block_w_start[0])
            reducer.flush()
            reducer.vectors_ready(lay.kv_b_start, lay.block_v_start[0])
            reducer.finish()
        self._last_grad_arena = garena
        # data parallel with `materialize_fp32=False`: the averaged weight gradients stay in the bf16 arena (read by
        # BridgeAdamW directly); the weights get no `.grad` until materialize_grads() is called
        lazy16 = reducer is not None and wgrad_bf16 and not reducer.materialize_fp32
        self._grad16 = g16 if lazy16 else None
        grads = []
        for name, p in self._named_params():
            o = lay.offsets[name]
            if p.requires_grad and not (lazy16 and o < lay.n_weights):
                grads.append(garena[o:o + p.numel()].view(p.shape))
            else:
                grads.append(None)
        d_text = d.view(B, L, D) if text_needs_grad else None
        return d_text, grads

    # -- public API ----------------------------------------------------------------------------------
    def forward(self, vision_features: torch.Tensor, text_embeddings: torch.Tensor, debug: bool = False,
                kv_cache=None, cached_positions: Optional[int] = None) -> torch.Tensor:
        """Same contract as the reference `BridgeLite.forward` (bridge_module.py:406-456).

        `kv_cache` (a `VisionKVCache`) is an additive, inference-only argument: when given, the
        per-image K/V projections are read from the cache instead of being recomputed.
        `cached_positions=k` (with `kv_cache`, eval mode) additionally declares that the first k text
        positions are the ones this cache last saw at those positions (a decode loop appending
        tokens): block 0's cross-attention rows of those positions are reused from the cache and
        only positions k.. are computed; k=0 (re)fills the cache from scratch.
        """
        params = [p for _, p in self._named_params()]
        needs_grad = torch.is_grad_enabled() and (text_embeddings.requires_grad or any(p.requires_grad for p in params))
        if vision_features is not None and vision_features.requires_grad and torch.is_grad_enabled():
            # the reference's vision encoder runs under no_grad (vision_encoder.py:89); this module has no
            # data-gradient kernel for the K/V projection and would silently hand back None
            raise RuntimeError("vision_features must not require grad: the bridge treats the image features as "
                               "constants (no gradient flows to the vision encoder)")
        if debug:
            return self._forward_debug(vision_features, text_embeddings, kv_cache)
        fp32 = kv_cache is not None and getattr(kv_cache, "precision", "bf16") == "fp32"
        if needs_grad:
            if kv_cache is not None or cached_positions is not None:
                raise RuntimeError("kv_cache is inference-only (use torch.no_grad())")
            return _BridgeFunction.apply(self, vision_features, text_embeddings, *params)
        if fp32:
            return self._run_forward_fp32(text_embeddings, kv_cache, cached_positions=cached_positions)
        out, _ = self._run_forward(vision_features, text_embeddings, keep_for_backward=False, kv_cache=kv_cache,
                                   cached_positions=cached_positions)
        return out      # fp32 like the reference's residual stream under autocast (SURVEY.md Appendix B)

    def materialize_grads(self) -> None:
        """Data parallel with `enable_data_parallel(..., materialize_fp32=False)`: turn the averaged bf16
        weight-gradient arena of the last backward into ordinary fp32 `.grad` tensors (one HBM-bound pass).
        `BridgeAdamW` does not need this; a loop that inspects or clips `.grad` itself does."""
        g16 = self.__dict__.get("_grad16")
        if g16 is None:
            return
        lay, garena = self._layout, self._last_grad_arena
        _lib.check(_lib.lib().b200b_bf16_to_f32(g16.data_ptr(), garena.data_ptr(), lay.n_weights, 1.0, _stream()),
                   "bf16_to_f32(materialize_grads)")
        for name, p in self._named_params():
            o = lay.offsets[name]
            if p.requires_grad and o < lay.n_weights:
                p.grad = garena[o:o + p.numel()].view(p.shape)
        self._grad16 = None

    def invalidate_weight_cache(self) -> None:
        """Force the bf16 operand copies to be re-made on the next call. The copies are refreshed when a
        parameter's version counter changes, which in-place autograd-visible updates (optimizers,
        `p.add_()`, `load_state_dict`) bump; writes through `p.data` (`p.data.copy_()`, EMA swaps, a custom
        broadcast, an external kernel writing the flat buffer) do not -- call this after any of those."""
        self._w16_key = None

    def _forward_debug(self, vision_features, text_embeddings, kv_cache):
        """debug=True: print the reference's per-block statistics (bridge_module.py:427-454).
        Runs the no-grad path per block, as the reference only uses it during generation."""
        print(f"🌉 Bridge Input - Vision: {vision_features.shape}, Text: {text_embeddings.shape}")
        print(f"    Text stats: mean={text_embeddings.mean():.4f}, std={text_embeddings.std():.4f}")
        print(f"    Vision stats: mean={vision_features.mean():.4f}, std={vision_features.std():.4f}")

        def cb(i, before, after):
            print(f"    Block {i + 1}: {before.mean():.4f}±{before.std():.4f} → {after.mean():.4f}±{after.std():.4f}")
            if torch.isnan(after).any():
                print(f"    ⚠️  NaN detected in Block {i + 1} output!")
            if torch.isinf(after).any():
                print(f"    ⚠️  Inf detected in Block {i + 1} output!")

        params = [p for _, p in self._named_params()]
        needs_grad = torch.is_grad_enabled() and (text_embeddings.requires_grad or any(p.requires_grad for p in params))
        if needs_grad:
            # keep autograd semantics; statistics are printed from a second, no-grad pass
            with torch.no_grad():
                was = self.training
                self.eval()
                self._run_forward(vision_features, text_embeddings, False, kv_cache, block_callback=cb)
                self.train(was)
            return _BridgeFunction.apply(self, vision_features, text_embeddings, *params)
        if kv_cache is not None and getattr(kv_cache, "precision", "bf16") == "fp32":
            return self._run_forward_fp32(text_embeddings, kv_cache, block_callback=cb)
        out, _ = self._run_forward(vision_features, text_embeddings, False, kv_cache, block_callback=cb)
        return out

    def get_model_info(self) -> dict:
        """Same keys as the reference (bridge_module.py:458-471)."""
        total_params = sum(p.numel() for p in self.parameters())
        trainable_params = sum(p.numel() for p in self.parameters() if p.requires_grad)
        return {
            "architecture": "Bridge-Lite",
            "num_blocks": self.num_blocks,
            "vision_dim": self.vision_dim,
            "language_dim": self.language_dim,
            "total_parameters": total_params,
            "trainable_parameters": trainable_params,
            "parameter_ratio": f"{trainable_params / total_params:.4f}",
        }
