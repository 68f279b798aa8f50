"""ctypes binding of the C-ABI library ``libfie_b200.so`` (declared in ``include/fie_b200.h``).

The product path has NO fallback: if the shared library is missing, cannot be loaded, or the device is not
sm_100, every op raises.  The library is built in-tree by ``csrc/build.sh`` (``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FIE_LIB") or os.path.join(_HERE, "libfie_b200.so")   # FIE_LIB: experiment builds only

DT_F16, DT_BF16, DT_F32 = 0, 1, 2       # out_dtype of the *_bf16 entry points (FIE_DT_*)

c_void_p, c_int, c_ll, c_float, c_size_t =ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_float, ctypes.c_size_t


class Epilogue(ctypes.Structure):
    """Mirror of ``fie_epilogue`` (include/fie_b200.h)."""
    _fields_ = [("col_bias", c_void_p), ("row_bias", c_void_p), ("rows_per_group", c_ll), ("ld_row_bias", c_ll), ("m_bias", c_void_p),
                ("residual", c_void_p), ("ld_res", c_ll), ("scale", c_float), ("act", c_int), ("out_f32", c_int),
                ("gn_stats", c_void_p), ("gn_groups", c_int), ("gn_rows_per_image", c_ll),
                ("ln_stats_out", c_void_p), ("ln_stats_in", c_void_p), ("ln_eps", c_float), ("ln_dim", c_int), ("row_scale", c_void_p)]


# name -> (restype, argtypes); must list every symbol include/fie_b200.h declares
SIGNATURES = {
    "fie_last_error": (ctypes.c_char_p, []),
    "fie_version": (c_int, []),
    "fie_device_supported": (c_int, []),
    "fie_canny_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "fie_canny_u8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "fie_rgb_to_gray_u8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "fie_gaussian_blur5_u8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "fie_jpeg_header_bytes": (c_int, []),
    "fie_jpeg_write_header": (c_int, [c_void_p, c_int, c_int, c_int]),
    "fie_jpeg_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "fie_jpeg_max_bytes": (c_size_t, [c_int, c_int]),
    "fie_jpeg_encode_u8": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p, c_void_p, c_size_t, c_void_p]),
    "fie_resample_lanczos_u8": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p]),
    "fie_ssim_u8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, ctypes.c_double, ctypes.c_double, ctypes.c_double, c_void_p, c_void_p]),
    "fie_sqdiff_u8": (c_int, [c_void_p, c_void_p, c_int, c_ll, c_void_p, c_void_p]),
    "fie_resample_f32": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int,
                                 c_void_p, c_void_p, c_void_p]),
    "fie_patchify_f16": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "fie_vit_assemble_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "fie_l2norm_rows_f16": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_ll, c_int, c_float, c_void_p]),
    "fie_sqdiff_f32": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_ll, c_int, c_void_p, c_void_p]),
    "fie_cosine_rows_f16": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_int, c_float, c_void_p]),
    "fie_im2col3x3_f16": (c_int, [c_void_p, c_int, c_ll, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "fie_maxpool3s2_ceil_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "fie_lpips_layer_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_ll, c_int, c_void_p, c_void_p]),
    "fie_preprocess_u8_to_f16_pad8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "fie_pad8_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "fie_postprocess_f16_to_u8": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p]),
    "fie_silu_f16": (c_int, [c_void_p, c_void_p, c_ll, c_void_p]),
    "fie_sincos_embedding": (c_int, [ctypes.POINTER(c_float), c_int, c_int, c_void_p, c_void_p]),
    "fie_softmax_rows_f32_to_f16": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_ll, c_int, c_float, c_void_p]),
    "fie_softmax_rows_f16": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_ll, c_int, c_float, c_void_p]),
    "fie_softmax_rows_exp_f16": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_int, c_float, c_void_p]),
    "fie_groupnorm_f16": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_ll, c_int, c_void_p, c_void_p, c_float, c_int, c_void_p, c_int, c_void_p]),
    "fie_layernorm_f16": (c_int, [c_void_p, c_void_p, c_ll, c_int, c_void_p, c_void_p, c_float, c_void_p]),
    "fie_geglu_block_n": (c_int, [c_int]),
    "fie_tune_gemm": (None, [c_int, c_int]),
    "fie_gemm_trace": (None, [c_void_p]),
    "fie_tune_conv_halo": (None, [c_int, c_int]),
    "fie_tune_conv_im2col": (None, [c_int]),
    "fie_tune_groupnorm_slab": (None, [c_int]),
    "fie_pack_conv3x3_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "fie_pack_conv3x3_c8_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "fie_pack_conv_up2x_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "fie_pack_rows_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "fie_fold_layernorm_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "fie_fuse_lora_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_float, c_int, c_int, c_ll, c_void_p]),
    "fie_gemm_f16": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_int, c_void_p, c_void_p, c_ll, c_ll, c_int, c_int, ctypes.POINTER(Epilogue), c_void_p]),
    "fie_conv3x3_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_ll, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(Epilogue), c_void_p]),
    "fie_conv_up2x_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_ll, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(Epilogue), c_void_p]),
    "fie_conv3x3_c8_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_ll, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(Epilogue), c_void_p]),
    "fie_conv3x3_cin4_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "fie_attn_vae_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "fie_attn_vae_d512_f16": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_void_p, c_ll, c_int, c_int, c_float, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "fie_attention_d64_f16": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "fie_attention_d64_causal_f16": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_ll, c_int, c_int, c_int, c_int, c_float, c_void_p]),
    "fie_embed_tokens_f16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_int, c_int, c_int, c_void_p]),
    "fie_gemm_bf16": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_int, c_void_p, c_void_p, c_ll, c_ll, c_int, c_int, ctypes.POINTER(Epilogue), c_int, c_void_p]),
    "fie_conv3x3_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_ll, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(Epilogue), c_int,
                                 c_void_p]),
    "fie_conv_up2x_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_ll, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(Epilogue), c_int, c_void_p]),
    "fie_conv3x3_c8_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_ll, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(Epilogue), c_int, c_void_p]),
    "fie_groupnorm_bf16_workspace_bytes": (c_size_t, [c_int, c_ll, c_int, c_int]),
    "fie_groupnorm_bf16": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_ll, c_int, c_void_p, c_void_p, c_float, c_int, c_void_p, c_size_t,
                                   c_void_p]),
    "fie_softmax_rows_f32_to_bf16": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_ll, c_int, c_float, c_void_p]),
    "fie_attn_vae_d512_bf16": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_void_p, c_void_p, c_ll, c_int, c_int, c_float, c_int, c_void_p, c_size_t, c_void_p]),
    "fie_pack_conv3x3_bf16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "fie_pack_conv_up2x_bf16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "fie_pack_rows_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "fie_canny_u8_per_image": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "fie_sincos_embedding_dev": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "fie_gemm_f16_ex": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_int, c_void_p, c_void_p, c_ll, c_ll, c_int, c_int, ctypes.POINTER(Epilogue), c_void_p,
                                c_void_p]),
    "fie_gemm_bf16_ex": (c_int, [c_void_p, c_ll, c_void_p, c_ll, c_int, c_void_p, c_void_p, c_ll, c_ll, c_int, c_int, ctypes.POINTER(Epilogue), c_int,
                                 c_void_p, c_void_p]),
    "fie_vae_sample_add_noise_batched": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_ll, c_float, c_void_p, c_void_p]),
    "fie_cfg_lcm_step_batched": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_ll, c_ll, c_void_p, c_int, c_void_p]),
}

_lib = None


class FieError(RuntimeError):
    pass


def build(verbose: bool = False) -> str:
    """Compile libfie_b200.so for sm_100a (nvcc cross-compiles without a GPU)."""
    out = subprocess.run(["bash", os.path.join(_HERE, "csrc", "build.sh")], capture_output=True, text=True)
    if out.returncode != 0:
        raise FieError("building libfie_b200.so failed:\n" + out.stdout + out.stderr)
    if verbose:
        print(out.stdout)
    return LIB_PATH


def lib() -> ctypes.CDLL:
    """Load (once) and return the C-ABI library; raises FieError if it is missing — there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FieError(f"{LIB_PATH} not found: run __graft_entry__.build() (csrc/build.sh). No CPU / PyTorch fallback exists.")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().fie_last_error().decode("utf-8", "replace")
        raise FieError(f"{what or 'fie call'} failed (rc={rc}): {msg}")
