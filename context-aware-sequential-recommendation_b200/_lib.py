"""ctypes binding of the C ABI declared in include/cast_b200.h.

The product path has exactly one backend: the sm_100a shared library built in-tree by `build.py`
(`csrc/libcast_b200.so`).  If it is missing, loading fails loudly — there is no CPU or PyTorch fallback.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libcast_b200.so")

P, L, I, F, U64, SZ = C.c_void_p, C.c_long, C.c_int, C.c_float, C.c_ulonglong, C.c_size_t

# name -> (restype, argtypes); mirrors include/cast_b200.h one to one
SIGNATURES = {
    "cast_version": (I, []),
    "cast_last_error_string": (C.c_char_p, []),
    "cast_launch_count": (U64, []),
    "cast_crc32c": (C.c_uint, [P, SZ, C.c_uint]),
    "cast_embed_fwd": (I, [P, P, I, I, L, I, F, P, P, F, U64, P, I, P, P, P]),
    "cast_mask_dropout": (I, [P, P, F, U64, P, I, L, I, P, P, P]),
    "cast_concat_dropout_fwd": (I, [P, I, I, L, I, F, I, F, I, U64, P, P, P]),
    "cast_concat_dropout_bwd": (I, [P, I, I, L, I, F, I, F, I, U64, P, P, P]),
    "cast_dropout_keep": (I, [F, U64, P, I, L, P, P]),
    "cast_add": (I, [P, P, P, L, P]),
    "cast_relu_bwd": (I, [P, P, F, P, L, P]),
    "cast_layernorm_fwd": (I, [P, P, P, L, I, F, P, P, P, P, P, P]),
    "cast_layernorm_bwd_workspace_bytes": (SZ, [L, I]),
    "cast_layernorm_bwd": (I, [P, P, P, P, P, L, I, P, P, P, P, P, SZ, P]),
    "cast_gemm_set_backend": (I, [I]),
    "cast_gemm_tensor_status": (I, [P, P]),
    "cast_gemm_workspace_bytes": (SZ, [L, I, L, I]),
    "cast_gemm": (I, [P, L, L, P, L, L, P, L, L, I, L, P, I, F, U64, P, I, P, L, F, P, L, P, I, P, SZ, P]),
    "cast_fused_supported": (I, [I]),
    "cast_ln_qkv_fwd": (I, [P, P, P, P, P, P, P, P, P, L, I, F, P, P, P, P, P, P, P, P, P]),
    "cast_ln_ffn_fwd": (I, [P, P, P, P, P, P, P, P, F, U64, P, I, I, L, I, F, P, P, P, P, P, P]),
    "cast_rowk_supported": (I, [I]),
    "cast_rowk_image_bytes": (SZ, [I]),
    "cast_rowk_presplit": (I, [P, I, I, P, SZ, P]),
    "cast_rowk_ln_qkv_fwd": (I, [P, P, P, P, P, P, P, L, I, F, P, P, P, P, P, P, P, P, P]),
    "cast_rowk_ln_ffn_fwd": (I, [P, P, P, P, P, P, P, F, U64, P, I, I, L, I, F, P, P, P, P, P, P]),
    "cast_rowk_status": (I, [P]),
    "cast_rowk_set_grid": (I, [I]),
    "cast_rowk_set_trace": (I, [P]),
    "cast_block_bwd_workspace_bytes": (SZ, [L, I]),
    "cast_ffn_bwd": (I, [P, P, P, P, P, P, P, P, P, P, F, U64, P, I, L, I, P, P, P, SZ, P]),
    "cast_qkv_bwd": (I, [P, P, P, P, P, P, P, P, P, P, P, P, L, I, P, P, P, SZ, P]),
    "cast_qkv_bwd_embed": (I, [P, P, P, P, P, P, P, P, P, P, P, P, L, I, P, F, U64, P, I, P, P, P, SZ, P]),
    "cast_colsum_workspace_bytes": (SZ, [L, L]),
    "cast_colsum": (I, [P, L, L, L, P, P, SZ, P]),
    "cast_attn_set_chunk": (I, [I]),
    "cast_set_pdl": (I, [I]),
    "cast_attn_set_kg": (I, [I]),
    "cast_fused_set_backend": (I, [I]),
    "cast_block_bwd_parts": (I, [L, I]),
    "cast_reduce_partials_batch": (I, [I, P, P, P, P, P, P]),
    "cast_layernorm_bwd_parts": (I, [L]),
    "cast_logits_loss_parts": (I, [L]),
    "cast_sampler_create": (P, [I, I, P, P, P, P, P, P, I, C.c_uint, P, I]),
    "cast_sampler_next": (I, [P, I, P, P, P, P, P, P, P, P]),
    "cast_sampler_next_raw": (I, [P, I, P, P, P, P, P]),
    "cast_sampler_destroy": (None, [P]),
    "cast_time_features": (I, [P, P, P, I, I, P, I, P, P, P, P]),
    "cast_lnf_loss_parts": (I, [L]),
    "cast_lnf_loss_workspace_bytes": (SZ, [L, I]),
    "cast_lnf_loss": (I, [P, P, P, F, P, I, I, L, P, P, P, P, P, P, P, P, P, SZ, P]),
    "cast_attn_fwd": (I, [P, L, P, L, P, L, P, P, P, I, I, I, I, F, U64, P, I, P, P, P, P, P, P]),
    "cast_attn_bwd": (I, [P, L, P, L, P, L, P, P, P, P, P, P, P, I, I, I, I, F, U64, P, I, P, L, P, L, P, L, P, P, P, SZ,
                      P]),
    "cast_attn_bwd_workspace_bytes": (SZ, [I, I, I]),
    "cast_logits_loss_workspace_bytes": (SZ, [L]),
    "cast_logits_loss": (I, [P, P, I, I, L, P, P, P, P, P, P, P, P, P, SZ, P]),
    "cast_scatter_workspace_bytes": (SZ, [L, I, I]),
    "cast_scatter_partial_bytes": (SZ, [L, I, I]),
    "cast_scatter_rows": (I, [P, I, L, P, P, P, I, I, P, P, SZ, P, SZ, P]),
    "cast_scatter_sort": (I, [P, I, L, I, P, SZ, P]),
    "cast_scatter_apply": (I, [I, L, P, P, P, I, I, P, P, SZ, P, SZ, I, P]),
    "cast_adam_init_state": (I, [P, F, F, P]),
    "cast_adam_tf_step": (I, [P, P, P, P, L, F, F, F, F, P, F, L, L, P, P]),
    "cast_adam_tf_range": (I, [P, P, P, P, L, F, F, F, F, P, F, L, L, P, I, P]),
    "cast_adam_tf_step_peers": (I, [P, P, I, P, P, P, L, L, F, F, F, F, F, L, L, P, P]),
    "cast_score_rank_cand": (I, [P, L, P, I, I, L, P, I, P, P, P, P]),
    "cast_score_rank_full_workspace_bytes": (SZ, [L, I, I]),
    "cast_score_rank_full": (I, [P, L, P, I, I, L, P, P, P, P, I, P, P, P, P, SZ, P]),
    "cast_embed_fwd_sharded": (I, [P, P, I, I, I, L, I, F, P, P, F, U64, P, I, P, P, P]),
    "cast_logits_loss_sharded": (I, [P, P, I, I, I, L, P, P, P, P, P, P, P, P, P, SZ, P]),
    "cast_score_rank_cand_sharded": (I, [P, L, P, I, I, I, L, P, I, P, P, P, P]),
    "cast_scatter_set_chunk": (I, [I]),
    "cast_scatter_sort_sharded": (I, [P, I, L, I, I, I, P, SZ, P]),
    "cast_scatter_sorted_offsets": (I, [L, I, I, P, P]),
    "cast_scatter_apply_range": (I, [I, L, P, P, P, I, P, P, P, C.c_uint, C.c_uint, P, SZ, I, P]),
    "cast_scatter_stage_bytes": (SZ, [L, I, I]),
    "cast_scatter_pull_range": (I, [I, L, P, P, P, I, P, P, P, C.c_uint, C.c_uint, P, SZ, P, SZ, I, P]),
    "cast_peer_alloc": (I, [SZ, P, P]),
    "cast_peer_free": (I, [P]),
    "cast_peer_open": (I, [P, P]),
    "cast_peer_close": (I, [P]),
    "cast_peer_barrier": (I, [P, I, I, P, P]),
    "cast_peer_reduce": (I, [P, I, L, P, P]),
    "cast_score_rank_full_status": (I, [P, L, I, P, P]),
    "cast_topk_full_workspace_bytes": (SZ, [L, I, I, I]),
    "cast_topk_full": (I, [P, L, P, I, I, L, I, P, P, I, P, P, P, P, SZ, P]),
    "cast_topk_full_status": (I, [P, L, I, I, I, P, P]),
}


class CastError(RuntimeError):
    pass


def bind(lib: C.CDLL) -> C.CDLL:
    """Attach restype/argtypes for every exported symbol; raises if one is missing."""
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:  # pragma: no cover
            raise CastError(f"{name} is not exported by {getattr(lib, '_name', lib)}") from e
        fn.restype = res
        fn.argtypes = args
    return lib


_LIB = None


def load_library(path: str | None = None) -> C.CDLL:
    """Loads the CUDA extension.  No fallback: a missing library is an error."""
    global _LIB
    if _LIB is not None and path is None:
        return _LIB
    p = path or LIB_PATH
    if not os.path.isfile(p):
        raise CastError(
            f"CUDA extension not found at {p}. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). This package has no CPU / PyTorch fallback.")
    lib = bind(C.CDLL(p))
    if os.environ.get("CAST_ATTN_CHUNK"):  # tuning hook (32 or 64 columns per streamed attention chunk)
        check(lib, lib.cast_attn_set_chunk(int(os.environ["CAST_ATTN_CHUNK"])), "cast_attn_set_chunk")
    if os.environ.get("CAST_PDL"):         # A/B hook: 0 = ordinary launches instead of programmatic dependent launch
        check(lib, lib.cast_set_pdl(int(os.environ["CAST_PDL"])), "cast_set_pdl")
    if os.environ.get("CAST_ATTN_KG"):     # tuning hook (2 or 4 key groups per row block of the attention kernels)
        check(lib, lib.cast_attn_set_kg(int(os.environ["CAST_ATTN_KG"])), "cast_attn_set_kg")
    if os.environ.get("CAST_FUSED_BACKEND"):  # A/B hook: 0 = FFMA row kernels, 1 = tensor-core row kernels
        check(lib, lib.cast_fused_set_backend(int(os.environ["CAST_FUSED_BACKEND"])), "cast_fused_set_backend")
    if path is None:
        _LIB = lib
    return lib


def check(lib: C.CDLL, rc: int, what: str = ""):
    if rc != 0:
        msg = lib.cast_last_error_string()
        raise CastError(f"{what} failed with code {rc}: {msg.decode() if msg else ''}")
