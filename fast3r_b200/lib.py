"""ctypes binding of libfast3r_b200.so (include/fast3r_b200.h).

There is NO fallback: if the library is missing or a call fails this raises (the reference's own native
precedent, curope, surfaces TORCH_CHECK failures as RuntimeError the same way —
fast3r/croco/models/curope/curope.cpp:54-59).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfast3r_b200.so")

EPI_STORE, EPI_ROPE, EPI_IDXEMB, EPI_CONVT, EPI_FINAL = range(5)
ACT_NONE, ACT_RELU, ACT_GELU = range(3)


class GemmDesc(C.Structure):
    _fields_ = [
        ("a", C.c_void_p), ("wt", C.c_void_p),
        ("n", C.c_int32), ("k", C.c_int32), ("taps", C.c_int32),
        ("w", C.c_int32), ("h", C.c_int32), ("nb", C.c_int32),
        ("a_ld", C.c_int32),
        ("epi", C.c_int32), ("act", C.c_int32),
        ("out0_f32", C.c_int32), ("res0_f32", C.c_int32),
        ("ldo", C.c_int32),
        ("split_col", C.c_int32), ("ldo_b", C.c_int32),
        ("tok_per_img", C.c_int32), ("grid_w", C.c_int32), ("rope_cols", C.c_int32),
        ("ct_k", C.c_int32), ("ct_cout", C.c_int32),
        ("bias", C.c_void_p), ("res0", C.c_void_p), ("res1", C.c_void_p),
        ("out0", C.c_void_p), ("out0b", C.c_void_p), ("out1", C.c_void_p),
        ("rope_cos", C.c_void_p), ("rope_sin", C.c_void_p),
        ("emb_table", C.c_void_p), ("emb_ids", C.c_void_p),
        ("w4", C.c_void_p), ("b4", C.c_void_p), ("pts", C.c_void_p), ("conf", C.c_void_p),
    ]


ABI_VERSION = 2
class BlockWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("norm1_w", "norm1_b", "norm2_w", "norm2_b", "qkv_w", "qkv_b", "proj_w", "proj_b",
                                          "fc1_w", "fc1_b", "fc2_w", "fc2_b")]


EXPORTS = ["f3r_last_error", "f3r_abi_version", "f3r_gemm_desc_size", "f3r_launch_count", "f3r_gemm", "f3r_attention",
           "f3r_layernorm", "f3r_im2col_patch", "f3r_im2col3x3s2", "f3r_upsample2x", "f3r_cast_bf16", "f3r_split3",
           "f3r_add_f32", "f3r_attention_x3_workspace", "f3r_attention_x3", "f3r_set_option", "f3r_attention_partial",
           "f3r_attention_merge", "f3r_resample_ksize", "f3r_resample_coeffs", "f3r_ingest_rgb8",
           "f3r_transformer_workspace", "f3r_transformer_blocks", "f3r_conf_quantile", "f3r_similarity_fit_workspace",
           "f3r_similarity_fit", "f3r_similarity_apply", "f3r_focal_workspace", "f3r_focal_weiszfeld",
           "f3r_pnp_workspace", "f3r_pnp_ransac"]

_lib = None


def load() -> C.CDLL:
    """Loads the shared library (no CUDA call is made); raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -m fast3r_b200.build` (or __graft_entry__.build()). "
            "fast3r_b200 has no CPU / PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    lib.f3r_last_error.restype = C.c_char_p
    lib.f3r_abi_version.restype = C.c_int
    lib.f3r_launch_count.restype = C.c_uint64
    lib.f3r_gemm.argtypes = [C.POINTER(GemmDesc), C.c_void_p]
    lib.f3r_attention_partial.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_float, C.c_void_p]
    lib.f3r_attention_merge.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                        C.c_int32, C.c_void_p]
    lib.f3r_attention_partial.restype = C.c_int
    lib.f3r_attention_merge.restype = C.c_int
    lib.f3r_resample_ksize.argtypes = [C.c_int32, C.c_int32, C.c_int32]
    lib.f3r_resample_ksize.restype = C.c_int
    lib.f3r_resample_coeffs.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    lib.f3r_resample_coeffs.restype = C.c_int
    lib.f3r_ingest_rgb8.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                    C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32,
                                    C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    lib.f3r_ingest_rgb8.restype = C.c_int
    lib.f3r_transformer_workspace.argtypes = [C.c_int32, C.c_int32, C.c_int32]
    lib.f3r_transformer_workspace.restype = C.c_size_t
    lib.f3r_transformer_blocks.argtypes = [C.POINTER(BlockWeights), C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                           C.c_int32, C.c_int32, C.c_float, C.c_float, C.c_int32, C.c_int32, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.f3r_transformer_blocks.restype = C.c_int
    lib.f3r_conf_quantile.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_void_p, C.c_void_p]
    lib.f3r_similarity_fit_workspace.argtypes = [C.c_int32]
    lib.f3r_similarity_fit_workspace.restype = C.c_size_t
    lib.f3r_similarity_fit.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                       C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.f3r_similarity_apply.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]
    lib.f3r_focal_workspace.argtypes = [C.c_int32]
    lib.f3r_focal_workspace.restype = C.c_size_t
    lib.f3r_focal_weiszfeld.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                        C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.f3r_pnp_workspace.argtypes = [C.c_int32] * 5
    lib.f3r_pnp_workspace.restype = C.c_size_t
    lib.f3r_pnp_ransac.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                   C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                   C.c_void_p]
    for name in ("f3r_conf_quantile", "f3r_similarity_fit", "f3r_similarity_apply", "f3r_focal_weiszfeld",
                 "f3r_pnp_ransac"):
        getattr(lib, name).restype = C.c_int
    lib.f3r_set_option.argtypes = [C.c_char_p, C.c_int32]
    lib.f3r_set_option.restype = C.c_int
    lib.f3r_attention.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
                                  C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_void_p]
    lib.f3r_layernorm.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                  C.c_float, C.c_void_p]
    lib.f3r_im2col_patch.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    lib.f3r_im2col3x3s2.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                    C.c_int32, C.c_void_p]
    lib.f3r_upsample2x.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_int32, C.c_int32, C.c_void_p]
    lib.f3r_split3.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int32, C.c_int32, C.c_void_p]
    lib.f3r_add_f32.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.f3r_attention_x3_workspace.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int32]
    lib.f3r_attention_x3_workspace.restype = C.c_size_t
    lib.f3r_attention_x3.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
                                     C.c_void_p, C.c_size_t, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float,
                                     C.c_void_p]
    lib.f3r_cast_bf16.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    for name in ("f3r_gemm", "f3r_attention", "f3r_layernorm", "f3r_im2col_patch", "f3r_im2col3x3s2",
                 "f3r_upsample2x", "f3r_cast_bf16", "f3r_split3", "f3r_add_f32", "f3r_attention_x3"):
        getattr(lib, name).restype = C.c_int
    lib.f3r_gemm_desc_size.restype = C.c_size_t
    if lib.f3r_abi_version() != ABI_VERSION or lib.f3r_gemm_desc_size() != C.sizeof(GemmDesc):
        raise RuntimeError("libfast3r_b200.so ABI mismatch (rebuild: python -m fast3r_b200.build --force)")
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise RuntimeError(f"fast3r_b200 {what} failed: {load().f3r_last_error().decode()}")


def set_option(name: str, value: int) -> None:
    check(load().f3r_set_option(name.encode(), int(value)), "f3r_set_option")


def launch_count() -> int:
    return int(load().f3r_launch_count())
