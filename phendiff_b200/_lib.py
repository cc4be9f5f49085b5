"""ctypes binding of libphendiff_b200.so (include/phendiff_b200.h).

There is deliberately NO fallback: if the shared library is missing or a call fails the product path raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libphendiff_b200.so"

PD_PREC_FP32, PD_PREC_BF16, PD_PREC_FP16 = 0, 1, 2
PD_PRED = {"epsilon": 0, "sample": 1, "v_prediction": 2}
PD_MAX_BLOCKS = 8


class UnetConfig(C.Structure):
    _fields_ = [
        ("in_channels", C.c_int32), ("out_channels", C.c_int32), ("n_blocks", C.c_int32),
        ("block_out_channels", C.c_int32 * PD_MAX_BLOCKS),
        ("down_attn", C.c_int32 * PD_MAX_BLOCKS), ("up_attn", C.c_int32 * PD_MAX_BLOCKS),
        ("layers_per_block", C.c_int32), ("attention_head_dim", C.c_int32), ("norm_num_groups", C.c_int32),
        ("norm_eps", C.c_float), ("num_class_embeds", C.c_int32), ("flip_sin_to_cos", C.c_int32),
        ("freq_shift", C.c_float), ("downsample_padding", C.c_int32), ("mid_block_scale_factor", C.c_float),
        ("add_attention", C.c_int32), ("precision", C.c_int32), ("max_microbatch", C.c_int32),
        ("conv_impl", C.c_int32), ("attn_impl", C.c_int32),
    ]


class StepCoeffs(C.Structure):
    _fields_ = [
        ("pred_type", C.c_int32), ("clip", C.c_int32), ("use_clipped_model_output", C.c_int32),
        ("clip_range", C.c_float), ("sqrt_alpha", C.c_float), ("sqrt_beta", C.c_float),
        ("sqrt_alpha_next", C.c_float), ("dir_coef", C.c_float), ("sigma", C.c_float), ("timestep", C.c_float),
    ]


class GradScalerState(C.Structure):
    """pd_grad_scaler_state_t: torch.amp.GradScaler's state, kept on the device by pd_adamw_step_scaled."""
    _fields_ = [("scale", C.c_float), ("growth_tracker", C.c_int32), ("optimizer_steps", C.c_int32), ("found_inf", C.c_int32),
                ("skipped_steps", C.c_int32)]


PD_ADAMW_SCRATCH_FLOATS = 1185
PD_ADAMW_SCALED_SCRATCH_FLOATS = 2376


class TestConvArgs(C.Structure):
    """pd_test_conv_args_t (kernel-level test entry point)."""
    _fields_ = ([(n, C.c_int32) for n in ("impl", "dtype", "n", "h", "w", "c1", "c2", "cout", "ksize", "stride", "pad", "upsample",
                                            "mode", "stats_cw", "csc1", "csc2")]
                + [(n, C.c_void_p) for n in ("x1", "x2", "weight", "bias", "addvec", "addvec_row", "residual", "sc1", "sc2", "sc_w")]
                + [("out_scale", C.c_float)]
                + [(n, C.c_void_p) for n in ("out", "stats_out", "model_out", "x_t", "step")])


_P = C.c_void_p
_SIGNATURES = {
    "pd_last_error": (C.c_char_p, []),
    "pd_version": (C.c_int, []),
    "pd_unet_create": (C.c_int, [C.POINTER(UnetConfig), C.POINTER(_P)]),
    "pd_unet_destroy": (C.c_int, [_P]),
    "pd_unet_num_params": (C.c_int, [_P, C.POINTER(C.c_int32)]),
    "pd_unet_param_info": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_char_p), C.POINTER(C.c_int32), C.POINTER(C.c_int64 * 4)]),
    "pd_unet_load_weight": (C.c_int, [_P, C.c_char_p, _P, C.POINTER(C.c_int64), C.c_int32]),
    "pd_unet_finalize": (C.c_int, [_P, _P]),
    "pd_unet_time_embed_dim": (C.c_int, [_P, C.POINTER(C.c_int32)]),
    "pd_unet_plan": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_size_t)]),
    "pd_unet_bind_workspace": (C.c_int, [_P, _P, C.c_size_t]),
    "pd_unet_forward": (C.c_int, [_P, _P, _P, _P, _P, _P, _P]),
    "pd_ddim_step": (C.c_int, [C.POINTER(StepCoeffs), _P, _P, _P, _P, _P, C.c_int64, _P]),
    "pd_axpby_per_sample": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, C.c_int64, _P]),
    "pd_cfg_combine": (C.c_int, [_P, _P, _P, C.c_int32, _P, C.c_int32, C.c_int64, _P]),
    "pd_denorm_nhwc": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P]),
    "pd_ddib_transfer": (C.c_int, [_P, _P, _P, _P, C.POINTER(StepCoeffs), C.c_int32, C.c_int32, _P]),
    "pd_unet_plan_guided": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_size_t)]),
    "pd_cfg_transfer": (C.c_int, [_P, _P, _P, _P, C.c_int32, C.POINTER(StepCoeffs), C.c_int32, _P]),
    "pd_train_create": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.POINTER(_P)]),
    "pd_train_destroy": (C.c_int, [_P]),
    "pd_train_set_precision": (C.c_int, [_P, C.c_int32]),
    "pd_train_set_loss_scale": (C.c_int, [_P, _P]),
    "pd_train_tc_counts": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "pd_train_num_params_flat": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "pd_train_param_offset": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int64)]),
    "pd_train_workspace_bytes": (C.c_int, [_P, C.POINTER(C.c_size_t)]),
    "pd_train_bind": (C.c_int, [_P, _P, C.c_size_t]),
    "pd_train_step_grad": (C.c_int, [_P] * 11),
    "pd_train_launch_count": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "pd_train_forward": (C.c_int, [_P] * 7),
    "pd_train_backward_input": (C.c_int, [_P] * 4),
    "pd_guidance_lp_grad": (C.c_int, [C.POINTER(StepCoeffs), _P, _P, _P, C.c_int32, C.c_int64, C.c_float, _P, _P, _P, _P, _P]),
    "pd_adamw_step": (C.c_int, [_P, _P, _P, _P, _P, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int32,
                                 C.c_float, C.c_float, _P, _P, _P]),
    "pd_adamw_step_scaled": (C.c_int, [_P, _P, _P, _P, _P, C.c_int64, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                                        C.c_float, _P, C.c_float, C.c_float, C.c_int32, _P, _P, _P]),
    "pd_debug_pair_kernel_launches": (C.c_longlong, []),
    "pd_unet_launch_count": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "pd_unet_plan_info": (C.c_int, [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "pd_unet_profile_begin": (C.c_int, [_P, C.c_int32, C.c_int32]),
    "pd_unet_profile_end": (C.c_int, [_P, C.POINTER(C.c_int32)]),
    "pd_unet_profile_query": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_double)]),
    "pd_unet_profile_op": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_char_p), C.POINTER(C.c_int32), C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_double)]),
    "pd_test_conv": (C.c_int, [C.c_int32] * 11 + [_P, _P, _P, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, C.c_float, _P, _P]),
    "pd_test_conv_ex": (C.c_int, [C.POINTER(TestConvArgs), _P]),
    "pd_test_gn_conv": (C.c_int, [C.c_int32] * 8 + [C.c_float] + [_P] * 10 + [C.c_int32, C.c_int32, _P, C.c_float, _P, _P, _P]),
    "pd_test_groupnorm": (C.c_int, [C.c_int32] * 6 + [C.c_float, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "pd_test_attention": (C.c_int, [C.c_int32] * 6 + [_P, _P, _P]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


class PhenDiffB200Error(RuntimeError):
    pass


def lib():
    """Load the shared library (once). Raises loudly when it is missing: there is no CPU / eager fallback."""
    global _lib
    if _lib is None:
        path = os.environ.get("PHENDIFF_B200_LIB", str(LIB_PATH))
        if not os.path.exists(path):
            raise PhenDiffB200Error(
                f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or phendiff_b200/csrc/build.sh). phendiff_b200 has no CPU or PyTorch fallback.")
        l = C.CDLL(path)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int):
    if rc != 0:
        msg = lib().pd_last_error()
        raise PhenDiffB200Error(msg.decode() if msg else f"phendiff_b200 error code {rc}")


def ptr(t):
    """Raw device pointer of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def current_stream():
    import torch

    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda(t, what: str):
    if not t.is_cuda:
        raise PhenDiffB200Error(
            f"{what} must be a CUDA tensor: phendiff_b200 is the B200 path and has no CPU fallback (got device {t.device})")
