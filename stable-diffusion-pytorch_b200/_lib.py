"""ctypes binding of the C-ABI kernel library (include/sdb200.h).

The library is built in-tree by ``build.py`` (nvcc, sm_100a) as
``stable-diffusion-pytorch_b200/libsdb200.so``.  Loading is lazy; every product
entry point goes through :func:`lib`, which raises if the library is missing —
there is no Python/CPU fallback for any kernel.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SDB200_LIB_PATH") or os.path.join(_HERE, "libsdb200.so")     # override: A/B experiments with another build

_lock = threading.Lock()
_lib = None

P, I64, I32, F32 = C.c_void_p, C.c_int64, C.c_int, C.c_float

# name -> argtypes; every function returns int (0 = ok) unless noted.  Kept in the same
# order as include/sdb200.h (tests/test_capi.py checks the two against each other).
SIGNATURES = {
    # --- sampler_kernels.cu
    "sdk_ddim_step": [P, P, P, F32, P, P, I64, P, I32, P, I64, I32, P],
    "sdk_ddpm_step": [P, P, P, F32, P, P, I64, P, I32, P, I64, P],
    "sdk_ddim_inpaint_step": [P, P, P, F32, P, I64, P, P, I64, I64, I64, P, I32, P, I64, I32, P],
    "sdk_ddpm_inpaint_step": [P, P, P, F32, P, I64, P, P, P, I64, I64, I64, P, I32, P, I64, P],
    "sdk_dpmpp_step": [P, P, P, F32, P, I32, P, I64, P, I32, P, I64, I32, P],
    "sdk_dpmpp_inpaint_step": [P, P, P, F32, P, I64, P, P, I64, I64, I64, P, I32, P, I64, I32, P, I32, P],
    "sdk_forward_process": [P, P, P, I64, I64, P, I32, P, P],
    "sdk_x0_from_eps": [P, P, F32, F32, P, I64, P],
    "sdk_next_timestep": [P, I32, P, P, P],
    "sdk_gather_row": [P, I64, I32, P, I32, P, P],
    # --- norm_kernels.cu
    "sdk_groupnorm_workspace_bytes": [I32, I32],
    "sdk_groupnorm_stats": [P, I32, P, I32, I32, I32, F32, P, P, P],
    "sdk_groupnorm_apply": [P, I32, P, I32, I32, I32, P, P, P, I32, P, P, I32, P],
    "sdk_groupnorm_apply_cs": [P, I32, P, P, I32, P, I32, I32, F32, P, P, I32, P, P, I32, P],
    "sdk_channel_stats": [P, I32, I32, I32, P, P],
    "sdk_conv_in": [P, P, P, P, P, I32, I32, I32, I32, P],
    "sdk_groupnorm_fused": [P, I32, P, I32, I32, I32, F32, P, P, I32, P, P, I32, P, P],
    "sdk_groupnorm_cluster": [P, I32, P, I32, I32, I32, F32, P, P, I32, P, P, I32, P],
    "sdk_layernorm": [P, P, P, F32, P, I32, I64, I32, P],
    "sdk_softmax_rows": [P, P, I32, I64, I32, F32, P],
    "sdk_embed_tokens": [P, P, P, P, I64, I32, I32, I32, P],
    "sdk_activation": [P, P, I32, I64, I32, P],
    "sdk_cast_upsample": [P, P, I32, I32, I32, I32, I32, I32, P],
    "sdk_nchw_to_nhwc": [P, P, I32, I32, I32, I32, P],
    # --- time_embed.cu
    "sdk_time_sinusoid": [P, I32, I32, P, P],
    "sdk_gemv": [P, I32, P, P, P, I32, I32, I32, I32, I32, P],
    # --- gemm_simt.cu
    "sdk_conv_gemm_f32": [P, P],
    # --- attention_simt.cu
    "sdk_attention_f32": [P, I64, I64, P, I64, I64, P, I64, I64, P, I64, I64, I32, I32, I32, I32, I32, F32, P],
    "sdk_attention_f32_ex": [P, I64, I64, P, I64, I64, P, I64, I64, P, I64, I64, I32, I32, I32, I32, I32, F32, I32, P],
    # --- attention_mma.cu
    "sdk_attention_bf16": [P, I64, I64, P, I64, I64, P, I64, I64, P, I64, I64, I32, I32, I32, I32, I32, F32, P],
    # --- attention_tc.cu
    "sdk_attention_tc_create": [P, I64, I64, P, I64, I64, P, I64, I64, P, I64, I64, I32, I32, I32, I32, I32, F32, P],
    "sdk_attention_tc_set_causal": [P, I32],
    "sdk_attention_tc_launch": [P, P],
    "sdk_attention_tc_destroy": [P],
    # --- gemm_tc.cu
    "sdk_tc_gemm_create": [P, P],
    "sdk_tc_gemm_workspace_bytes": [P],
    "sdk_tc_gemm_set_workspace": [P, P],
    "sdk_tc_gemm_info": [P, P, I32],
    "sdk_tc_gemm_launch": [P, P],
    "sdk_tc_gemm_destroy": [P],
    "sdk_tc_gemm_set_debug": [P, P],
    "sdk_tc_gemm_set_stats": [P, P],
    "sdk_zero": [P, I64, P],
    "sdk_im2col_s2": [P, P, I32, I32, I32, I32, P],
    # --- linear_ln.cu
    "sdk_linear_ln_create": [P, P],
    "sdk_linear_ln_info": [P, P, I32],
    "sdk_linear_ln_launch": [P, P],
    "sdk_linear_ln_destroy": [P],
    # --- lora_merge.cu
    "sdk_lora_merge": [P, I64, P, P, I32, P, I32, I32, I32, I32, I32, I32, I32, P],
    # --- plan.cu
    "sdk_plan_create": [P],
    "sdk_plan_destroy": [P],
    "sdk_plan_add_region": [P, P, I64, I32, C.c_char_p],
    "sdk_plan_adopt": [P, I32, P, P, I32, P, I32],
    "sdk_plan_add_launch": [P, I32, C.c_char_p, P, I32],
    "sdk_plan_num_launches": [P, I32],
    "sdk_plan_launch": [P, I32, P],
    "sdk_plan_capture": [P, I32, P],
    "sdk_plan_save": [P, C.c_char_p],
    "sdk_plan_load": [C.c_char_p, P],
    "sdk_plan_region": [P, C.c_char_p, P, P],
    "sdk_plan_upload": [P, C.c_char_p, P, I64, P],
    "sdk_plan_download": [P, C.c_char_p, P, I64, P],
    "sdk_stream_create": [P],
    "sdk_stream_sync": [P],
    "sdk_stream_destroy": [P],
    # --- misc
    "sdk_device_info": [P, I32],
    "sdk_set_pdl": [I32],
    "sdk_set_uniform_carveout": [I32],
}


class ConvParams(C.Structure):
    """Mirror of SdkConvParams (include/sdb200.h)."""
    _fields_ = [("src0", P), ("src1", P), ("weight", P), ("bias", P), ("tbias", P), ("residual", P), ("out", P),
                ("tb_stride", I64), ("C0", I32), ("C1", I32),
                ("B", I32), ("Hin", I32), ("Win", I32), ("Hout", I32), ("Wout", I32),
                ("ksize", I32), ("stride", I32), ("upsample", I32), ("N", I32),
                ("in_dtype", I32), ("out_dtype", I32), ("out_nchw", I32), ("geglu", I32)]


class TcGemmDesc(C.Structure):
    """Mirror of SdkTcGemmDesc (include/sdb200.h)."""
    _fields_ = [("a", P * 2), ("w", P * 2), ("C", I32 * 2), ("ksize", I32 * 2), ("nseg", I32),
                ("B", I32), ("H", I32), ("W", I32), ("N", I32),
                ("bias", P), ("tbias", P), ("tb_stride", I64), ("residual", P), ("out", P),
                ("out_dtype", I32), ("geglu", I32), ("out_nchw", I32), ("block_n", I32), ("splits", I32), ("w_kmajor", I32), ("two_cta", I32),
                ("out2", P), ("row_stats", P), ("ln_stats", P), ("ln_colsum", P), ("ln_parts", I32), ("ln_eps", F32),
                ("a_stride", I32), ("a_h", I32), ("a_w", I32), ("up2", I32), ("w_const", I32), ("weight_stationary", I32)]


class LinearLnDesc(C.Structure):
    """Mirror of SdkLinearLnDesc (include/sdb200.h)."""
    _fields_ = [("a", P), ("w", P), ("bias", P), ("residual", P), ("out", P), ("ln_out", P), ("gamma", P), ("beta", P),
                ("eps", F32), ("M", I64), ("K", I32), ("N", I32)]


class AttentionTcDesc(C.Structure):
    """Mirror of SdkAttentionTcDesc (include/sdb200.h)."""
    _fields_ = [("q", P), ("k", P), ("v", P), ("out", P),
                ("q_row", I64), ("q_batch", I64), ("k_row", I64), ("k_batch", I64), ("v_row", I64), ("v_batch", I64),
                ("o_row", I64), ("o_batch", I64), ("B", I32), ("heads", I32), ("Sq", I32), ("Sk", I32), ("D", I32), ("scale", F32)]


F32_T, BF16_T = 0, 1
RESTYPES = {"sdk_last_error": C.c_char_p, "sdk_version": C.c_int, "sdk_groupnorm_workspace_bytes": C.c_int64,
            "sdk_tc_gemm_workspace_bytes": C.c_int64}
SIGNATURES.update({"sdk_last_error": [], "sdk_version": []})


class ExtensionMissing(RuntimeError):
    pass


def lib():
    """The loaded C-ABI library; raises ExtensionMissing if it was never built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise ExtensionMissing(
                    f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                    "(nvcc, sm_100a). The B200 path has no CPU/PyTorch fallback.")
            h = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
            for name, argtypes in SIGNATURES.items():
                fn = getattr(h, name)          # AttributeError here == header/library drift
                fn.argtypes = argtypes
                fn.restype = RESTYPES.get(name, C.c_int)
            h.sdk_set_pdl(0 if os.environ.get("SDB200_PDL", "1") == "0" else 1)     # programmatic dependent launch: measured 4.29 -> 4.15 ms/step (round 2)
            h.sdk_set_uniform_carveout(1 if os.environ.get("SDB200_UNIFORM_CARVEOUT", "0") == "1" else 0)
            _lib = h
    return _lib


def check(status: int):
    if status != 0:
        msg = lib().sdk_last_error()
        raise RuntimeError(f"sdb200 kernel library error {status}: {msg.decode() if msg else '?'}")


def current_stream(device) -> int:
    """cudaStream_t of torch's current stream on ``device`` (what every launch is enqueued on)."""
    return torch.cuda.current_stream(device).cuda_stream
