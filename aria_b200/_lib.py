"""ctypes binding of libaria_b200.so (the C ABI declared in include/aria_b200.h).

There is no fallback: if the shared library is missing or a call fails, we raise.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# ARIA_B200_LIB selects another build of the same C ABI (kernel A/B experiments); default: the in-tree build
LIB_PATH = os.environ.get("ARIA_B200_LIB") or os.path.join(_HERE, "libaria_b200.so")

ARIA_OK = 0
B_NK, B_GKN, B_GNK = 0, 1, 2
EPI_LINEAR, EPI_SWIGLU, EPI_HEADS = 0, 1, 2
ACT_NONE, ACT_GELU_TANH, ACT_GELU_NEW = 0, 1, 2

_ERR = {-1: "bad argument", -2: "unsupported shape", -3: "CUDA error"}

vp = C.c_void_p
i32 = C.c_int32
i64 = C.c_int64
f32 = C.c_float


class GemmDesc(C.Structure):
    """Mirror of `aria_gemm_desc_t` (include/aria_b200.h) — keep field order in sync."""

    _fields_ = [
        ("a", vp), ("lda", i64), ("m", i64), ("n", i64), ("k", i64),
        ("b", vp * 3), ("n_seg", i32), ("b_layout", i32),
        ("num_groups", i32), ("group_offsets", vp), ("group_mod", i32),
        ("epilogue", i32), ("act", i32),
        ("bias", vp * 3), ("residual", vp), ("ldr", i64),
        ("out", vp * 3), ("ldo", i64),
        ("head_dim", i32), ("head_ld", i32), ("rows_per_batch", i32), ("pos0", i32),
        ("stride_b", i64), ("stride_h", i64),
        ("rope_mask", i32), ("rope_cos", vp), ("rope_sin", vp), ("position_ids", vp),
        ("dbg_lbo", i32), ("dbg_sbo", i32), ("dbg_kadv", i32),
        ("group_counts", vp), ("a_rows", i64), ("out_group_base", vp), ("out_group_row0", vp),
    ]


# symbol -> (restype, argtypes); this table is also what tests/test_abi.py checks against the header.
SIGNATURES = {
    "aria_abi_version": (i32, []),
    "aria_build_arch": (C.c_char_p, []),
    "aria_gemm": (i32, [C.POINTER(GemmDesc), vp]),
    "aria_grouped_gemm": (i32, [vp, vp, vp, vp, i64, i64, i64, i32, vp]),
    "aria_offsets_from_counts": (i32, [vp, vp, i32, vp]),
    "aria_router_topk": (i32, [vp, vp, vp, vp, vp, vp, i64, i32, i32, i32, vp]),
    "aria_route_from_logits": (i32, [vp, vp, vp, vp, i64, i32, i32, vp]),
    "aria_route_given_indices": (i32, [vp, vp, vp, vp, i64, i32, i32, vp]),
    "aria_build_permutation": (i32, [vp, vp, vp, vp, vp, i64, i32, i32, i32, vp]),
    "aria_grouped_wgrad": (i32, [vp, i64, vp, i64, vp, vp, i64, i64, i64, i32, i32, vp]),
    "aria_moe_block_fwd_workspace_bytes": (i64, [i64, i32, i32, i32, i32, i32]),
    "aria_moe_block_fwd": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, i64, i32, i32, i32, i32, i32, vp, vp, i64, vp, vp]),
    "aria_swiglu_fwd": (i32, [vp, vp, i64, i32, vp]),
    "aria_swiglu_bwd": (i32, [vp, vp, vp, i64, i32, vp]),
    "aria_combine_bwd": (i32, [vp, vp, vp, vp, vp, vp, i64, i32, i32, vp]),
    "aria_router_bwd": (i32, [vp, vp, vp, vp, i64, i32, i32, vp]),
    "aria_router_aux_workspace_bytes": (C.c_size_t, [i32]),
    "aria_router_aux_loss": (i32, [vp, vp, vp, i64, i32, i32, f32, f32, vp, C.c_size_t, vp]),
    "aria_router_aux_bwd": (i32, [vp, vp, vp, i64, i32, i32, f32, f32, f32, vp]),
    "aria_permute_rows": (i32, [vp, vp, vp, i64, i32, vp]),
    "aria_unpermute_combine": (i32, [vp, vp, vp, vp, vp, i64, i32, i32, vp]),
    "aria_rmsnorm": (i32, [vp, vp, vp, vp, vp, i64, i32, f32, vp]),
    "aria_layernorm": (i32, [vp, vp, vp, vp, i64, i32, f32, vp]),
    "aria_rope_table": (i32, [vp, vp, vp, i32, i32, vp]),
    "aria_embedding": (i32, [vp, vp, vp, i64, i32, vp]),
    "aria_merge_image_features": (i32, [vp, i64, vp, vp, vp, i64, i32, vp]),
    "aria_im2col_patches": (i32, [vp, vp, i32, i32, i32, i32, vp]),
    "aria_add_pos_embedding": (i32, [vp, vp, vp, vp, i64, i32, vp]),
    "aria_enable_peer_access": (i32, [i32]),
    "aria_ipc_export": (i32, [vp, vp, vp]),
    "aria_ipc_open": (i32, [vp, vp]),
    "aria_ipc_close": (i32, [vp]),
    "aria_ep_publish_counts": (i32, [vp, vp, i32, i32, i32, vp]),
    "aria_peer_barrier": (i32, [vp, i32, i32, vp, vp]),
    "aria_ep_layout": (i32, [vp, i32, i32, i32, vp, vp, vp, vp]),
    "aria_scatter_rows_grouped": (i32, [vp, vp, vp, i32, vp, i32, vp, i32, i64, vp]),
    "aria_ep_dispatch": (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i64, vp]),
    "aria_attention_fwd": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, i64, i64, i64, i64, i32, f32, i32, vp, i64, vp]),
    "aria_attention_fwd_workspace_bytes": (i64, [i32, i32, i32, i32, i32, i32]),
    "aria_attention_decode": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i64, i64, i64, i64, f32, vp, i64, vp]),
    "aria_attention_decode_workspace_bytes": (i64, [i32, i32, i32]),
    "aria_attention_fwd_lse": (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, i64, i64, i64, i64, f32, i32, i32, vp]),
    "aria_attention_bwd_workspace_bytes": (i64, [i32, i32, i32]),
    "aria_attention_bwd": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i64, i64, i64, i64, f32, i32, i32, vp, i64,
                                 vp]),
    "aria_rmsnorm_bwd_workspace_bytes": (i64, [i64, i32]),
    "aria_rmsnorm_bwd": (i32, [vp, vp, vp, vp, vp, vp, i64, i32, f32, vp, i64, vp]),
    "aria_rope_bwd": (i32, [vp, vp, vp, vp, i64, i32, i32, vp]),
    "aria_lm_xent_fwd_workspace_bytes": (i64, [i64, i64]),
    "aria_lm_xent_fwd": (i32, [vp, vp, vp, vp, vp, vp, i64, i64, i32, vp, i64, vp]),
    "aria_lm_xent_bwd_workspace_bytes": (i64, [i64, i64, i32]),
    "aria_lm_xent_bwd": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, i64, i64, i32, vp, i64, vp]),
    "aria_embedding_bwd_workspace_bytes": (i64, [i64, i64]),
    "aria_embedding_bwd": (i32, [vp, vp, vp, i64, i32, i64, i64, vp, i64, vp]),
}

_lib = None


def load():
    """Load the shared library (once). Raises if it has not been built — no silent fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -m aria_b200.build` (nvcc, sm_100a). "
            "aria_b200 has no CPU/eager fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in list(SIGNATURES.items()) + list(EXTRA_SIGNATURES.items()):
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


# kernels launched per C-ABI call (for bench.py's `gpu_launches`; memsets are not counted)
KERNELS_PER_CALL = {"router_topk": 2, "attention_decode": 2, "moe_block_fwd": 9, "attention_bwd": 3, "rmsnorm_bwd": 2,
                    "lm_xent_fwd": 3, "embedding_bwd": 4}
# kernels exported for A/B measurements only (scripts/), not part of include/aria_b200.h
EXTRA_SIGNATURES = {
    "aria_attention_fwd_v2": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, i64, i64, i64, i64, i32, f32, i32, vp]),
}
launch_count = 0


def check(rc: int, what: str):
    global launch_count
    if rc != ARIA_OK:
        raise RuntimeError(f"aria_b200: {what} failed: {_ERR.get(rc, rc)}")
    launch_count += KERNELS_PER_CALL.get(what, 1)
