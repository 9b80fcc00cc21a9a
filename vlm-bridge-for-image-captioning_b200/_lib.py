"""ctypes binding of libb200_bridge.so (C ABI declared in include/b200_bridge.h).

There is no CPU fallback: if the shared library is missing or a call fails, a RuntimeError is
raised. `torch` is only used by callers for device memory and streams; no torch type crosses the
ABI (plain pointers and sizes).
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "csrc", "libb200_bridge.so")

# enum b200b_epilogue
EPI_BF16_BIAS = 0
EPI_BF16_BIAS_GELU = 1
EPI_F32_BIAS_RESID = 2
EPI_BF16_DGELU = 3
EPI_F32 = 4
NVLS_OUT_MULTICAST = 1      # B200B_NVLS_OUT_MULTICAST
NVLS_EXCLUSIVE_SMS = 2      # B200B_NVLS_EXCLUSIVE_SMS


class GemmArgs(C.Structure):
    _fields_ = [
        ("a", C.c_void_p),
        ("b", C.c_void_p),
        ("a_major", C.c_int32),
        ("b_major", C.c_int32),
        ("m", C.c_int32),
        ("n", C.c_int32),
        ("k", C.c_int32),
        ("lda", C.c_int64),
        ("ldb", C.c_int64),
        ("epilogue", C.c_int32),
        ("block_n", C.c_int32),
        ("out", C.c_void_p),
        ("ldo", C.c_int64),
        ("aux", C.c_void_p),
        ("ldaux", C.c_int64),
        ("bias", C.c_void_p),
        ("resid", C.c_void_p),
        ("ldr", C.c_int64),
        ("beta", C.c_float),
        ("dropout_p", C.c_float),
        ("seed", C.c_uint64),
        ("dropout_stream", C.c_uint32),
        ("cta_group", C.c_uint32),
    ]


class ColsumTask(C.Structure):
    _fields_ = [("partials", C.c_void_p), ("out", C.c_void_p), ("cols", C.c_int32), ("chunks", C.c_int32),
                ("chunk_stride", C.c_int64)]


class NvlsComm(C.Structure):
    _fields_ = [("multicast_base", C.c_void_p), ("local_base", C.c_void_p), ("flags", C.c_void_p * 8),
                ("rank", C.c_int32), ("world", C.c_int32), ("timeout_s", C.c_int32), ("reserved", C.c_int32),
                ("error_word", C.c_void_p)]


class BeamState(C.Structure):
    """b200b_beam_state"""
    _fields_ = [("beam_scores", C.c_void_p), ("hyp_scores", C.c_void_p), ("hyp_lens", C.c_void_p),
                ("hyp_seq", C.c_void_p), ("hyp_count", C.c_void_p), ("done", C.c_void_p), ("hyp_ids", C.c_void_p),
                ("ld_hyp", C.c_int64)]


class AttnArgs(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("ldq", C.c_int64),
        ("k", C.c_void_p), ("ldk", C.c_int64),
        ("v", C.c_void_p), ("ldv", C.c_int64),
        ("o", C.c_void_p), ("ldo", C.c_int64),
        ("lse", C.c_void_p),
        ("d_o", C.c_void_p), ("lddo", C.c_int64),
        ("dq", C.c_void_p), ("lddq", C.c_int64),
        ("dk", C.c_void_p), ("lddk", C.c_int64),
        ("dv", C.c_void_p), ("lddv", C.c_int64),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_uint64),
        ("batch", C.c_int32), ("heads", C.c_int32), ("len_q", C.c_int32), ("len_k", C.c_int32),
        ("head_dim", C.c_int32),
        ("dropout_p", C.c_float),
        ("seed", C.c_uint64),
        ("dropout_stream", C.c_uint32),
        ("reserved", C.c_uint32),
    ]


_lock = threading.Lock()
_lib = None


def _declare(lib) -> None:
    lib.b200b_abi_version.restype = C.c_int
    lib.b200b_abi_version.argtypes = []
    lib.b200b_last_error.restype = C.c_char_p
    lib.b200b_last_error.argtypes = []
    lib.b200b_launch_count.restype = C.c_uint64
    lib.b200b_launch_count.argtypes = []
    lib.b200b_profile_begin.restype = C.c_int
    lib.b200b_profile_begin.argtypes = [C.c_void_p]
    lib.b200b_profile_end.restype = C.c_int
    lib.b200b_profile_end.argtypes = []
    lib.b200b_profile_entry.restype = C.c_char_p
    lib.b200b_profile_entry.argtypes = [C.c_int, C.POINTER(C.c_float)]
    lib.b200b_gemm.restype = C.c_int
    lib.b200b_gemm.argtypes = [C.POINTER(GemmArgs), C.c_void_p]
    lib.b200b_layernorm_fwd.restype = C.c_int
    lib.b200b_layernorm_fwd.argtypes = [C.c_void_p] * 6 + [C.c_int, C.c_int, C.c_float, C.c_void_p]
    lib.b200b_layernorm_bwd.restype = C.c_int
    lib.b200b_layernorm_bwd.argtypes = [C.c_void_p] * 7 + [C.c_int, C.c_int, C.c_void_p]
    lib.b200b_colsum_workspace_bytes.restype = C.c_size_t
    lib.b200b_colsum_workspace_bytes.argtypes = [C.c_int, C.c_int]
    lib.b200b_colsum.restype = C.c_int
    lib.b200b_colsum.argtypes = [C.c_void_p, C.c_int64] + [C.c_void_p] * 5 + [C.c_int, C.c_int, C.c_void_p,
                                                                               C.c_size_t, C.c_void_p]
    lib.b200b_cast_bf16.restype = C.c_int
    lib.b200b_cast_bf16.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_uint64, C.c_uint32,
                                    C.c_void_p]
    lib.b200b_row_chunks.restype = C.c_int
    lib.b200b_row_chunks.argtypes = [C.c_int]
    lib.b200b_layernorm_fwd_rows.restype = C.c_int
    lib.b200b_layernorm_fwd_rows.argtypes = [C.c_void_p] * 6 + [C.c_int, C.c_int, C.c_float, C.c_void_p]
    lib.b200b_layernorm_bwd_fused.restype = C.c_int
    lib.b200b_layernorm_bwd_fused.argtypes = [C.c_void_p] * 9 + [C.c_int, C.c_int, C.c_void_p]
    lib.b200b_cast_bf16_colsum.restype = C.c_int
    lib.b200b_cast_bf16_colsum.argtypes = [C.c_void_p] * 3 + [C.c_int, C.c_int, C.c_float, C.c_uint64, C.c_uint32,
                                           C.c_void_p]
    lib.b200b_colsum_partials.restype = C.c_int
    lib.b200b_colsum_partials.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int),
                                          C.c_void_p]
    lib.b200b_bf16_to_f32.restype = C.c_int
    lib.b200b_bf16_to_f32.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_void_p]
    lib.b200b_allreduce_nvls_flag_bytes.restype = C.c_size_t
    lib.b200b_allreduce_nvls_flag_bytes.argtypes = []
    lib.b200b_allreduce_nvls.restype = C.c_int
    lib.b200b_allreduce_nvls.argtypes = [C.POINTER(NvlsComm), C.c_int, C.c_int64, C.c_int64, C.c_float, C.c_void_p,
                                         C.c_uint32, C.c_void_p, C.c_int, C.c_int, C.c_uint32, C.c_void_p]
    lib.b200b_grad_sqnorm_workspace_bytes.restype = C.c_size_t
    lib.b200b_grad_sqnorm_workspace_bytes.argtypes = []
    lib.b200b_grad_sqnorm.restype = C.c_int
    lib.b200b_grad_sqnorm.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
    lib.b200b_adamw_fused.restype = C.c_int
    lib.b200b_adamw_fused.argtypes = [C.c_void_p] * 6 + [C.c_int64, C.c_int64, C.c_void_p, C.c_float, C.c_void_p,
                                                          C.c_void_p] + [C.c_float] * 5 + [C.c_int64, C.c_void_p, C.c_void_p]
    lib.b200b_cross_entropy_fwd.restype = C.c_int
    lib.b200b_cross_entropy_fwd.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p] + [C.c_int64] * 4 + [C.c_void_p] * 4
    lib.b200b_cross_entropy_bwd.restype = C.c_int
    lib.b200b_cross_entropy_bwd.argtypes = ([C.c_void_p, C.c_int, C.c_int64, C.c_void_p] + [C.c_int64] * 4 +
                                            [C.c_void_p] * 4 + [C.c_int64, C.c_void_p])
    lib.b200b_sample_tokens.restype = C.c_int
    lib.b200b_sample_tokens.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_float, C.c_float,
                                        C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
    lib.b200b_sample_tokens_top_k.restype = C.c_int
    lib.b200b_sample_tokens_top_k.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_float, C.c_int64,
                                              C.c_float, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
    lib.b200b_beam_step_workspace_bytes.restype = C.c_size_t
    lib.b200b_beam_step_workspace_bytes.argtypes = [C.c_int64, C.c_int]
    lib.b200b_beam_step.restype = C.c_int
    lib.b200b_beam_step.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int, C.c_int64, C.c_int64, C.c_float,
                                    C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                    C.POINTER(BeamState), C.c_void_p, C.c_size_t, C.c_void_p]
    lib.b200b_beam_finalize.restype = C.c_int
    lib.b200b_beam_finalize.argtypes = [C.c_int64, C.c_int, C.c_int64, C.c_float, C.c_int64, C.c_void_p, C.c_int64,
                                        C.POINTER(BeamState), C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                        C.c_void_p]
    lib.b200b_beam_finalize_top.restype = C.c_int
    lib.b200b_beam_finalize_top.argtypes = [C.c_int64, C.c_int, C.c_int, C.c_int64, C.c_float, C.c_int64, C.c_void_p,
                                            C.c_int64, C.POINTER(BeamState), C.c_void_p, C.c_int64, C.c_void_p,
                                            C.c_void_p, C.c_void_p]
    lib.b200b_gemm_dual.restype = C.c_int
    lib.b200b_gemm_dual.argtypes = [C.POINTER(GemmArgs), C.POINTER(GemmArgs), C.c_void_p]
    lib.b200b_gemm_set_dual.restype = C.c_int
    lib.b200b_gemm_set_dual.argtypes = [C.c_int]
    lib.b200b_attention_set_tc.restype = C.c_int
    lib.b200b_attention_set_tc.argtypes = [C.c_int]
    lib.b200b_set_sm_limit.restype = None
    lib.b200b_set_sm_limit.argtypes = [C.c_int]
    lib.b200b_get_sm_limit.restype = C.c_int
    lib.b200b_get_sm_limit.argtypes = []
    lib.b200b_colsum_finalize.restype = C.c_int
    lib.b200b_colsum_finalize.argtypes = [C.POINTER(ColsumTask), C.c_int, C.c_void_p]
    lib.b200b_attention_fwd.restype = C.c_int
    lib.b200b_attention_fwd.argtypes = [C.POINTER(AttnArgs), C.c_void_p]
    lib.b200b_kv_cache_packed_bytes.restype = C.c_size_t
    lib.b200b_kv_cache_packed_bytes.argtypes = [C.c_int] * 5
    lib.b200b_kv_cache_pack.restype = C.c_int
    lib.b200b_kv_cache_pack.argtypes = [C.c_void_p, C.c_int64, C.c_void_p] + [C.c_int] * 5 + [C.c_void_p]
    lib.b200b_attention_decode_packed.restype = C.c_int
    lib.b200b_attention_decode_packed.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                                  C.c_int64, C.c_void_p] + [C.c_int] * 5 + [C.c_void_p]
    lib.b200b_kv_cache_tc_bytes.restype = C.c_size_t
    lib.b200b_kv_cache_tc_bytes.argtypes = [C.c_int] * 5
    lib.b200b_kv_cache_pack_tc.restype = C.c_int
    lib.b200b_kv_cache_pack_tc.argtypes = [C.c_void_p, C.c_int64, C.c_void_p] + [C.c_int] * 5 + [C.c_void_p]
    lib.b200b_attention_decode_tc.restype = C.c_int
    lib.b200b_attention_decode_tc.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                              C.c_int64, C.c_void_p] + [C.c_int] * 5 + [C.c_void_p]
    lib.b200b_attention_bwd_workspace_bytes.restype = C.c_size_t
    lib.b200b_attention_bwd_workspace_bytes.argtypes = [C.c_int] * 4
    lib.b200b_attention_bwd.restype = C.c_int
    lib.b200b_attention_bwd.argtypes = [C.POINTER(AttnArgs), C.c_void_p]


def lib():
    """Load (once) and return the shared library; raise if it has not been built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        f"{LIB_PATH} is missing: build it with `python -m vlm_bridge_b200.build` "
                        "(there is no CPU or PyTorch fallback for the bridge kernels)"
                    )
                handle = C.CDLL(LIB_PATH)
                _declare(handle)
                _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().b200b_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"b200b {what} failed (rc={rc}): {msg}")


def launch_count() -> int:
    return int(lib().b200b_launch_count())


def profile_begin(stream_ptr: int) -> None:
    check(lib().b200b_profile_begin(C.c_void_p(stream_ptr)), "profile_begin")


def profile_end() -> list[tuple[str, float]]:
    """[(kernel name, milliseconds)] of every launch since profile_begin()."""
    n = lib().b200b_profile_end()
    out = []
    ms = C.c_float()
    for i in range(n):
        name = lib().b200b_profile_entry(i, C.byref(ms))
        if name is None:
            break
        out.append((name.decode(), float(ms.value)))
    return out
