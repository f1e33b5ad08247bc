"""ctypes binding of libdiamond_b200.so (C ABI: include/diamond_b200.h)."""
import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdiamond_b200.so")
DMD_MAX_LEVELS = 8

_vp, _i, _f, _sz = C.c_void_p, C.c_int, C.c_float, C.c_size_t


class PrepDesc(C.Structure):
    _fields_ = [
        ("src0", _vp), ("src1", _vp), ("C0", _i), ("C1", _i), ("B", _i), ("Hs", _i), ("Ws", _i), ("upsample", _i),
        ("mode", _i), ("silu", _i), ("stats0", _vp), ("stats1", _vp), ("gs0", _i), ("gs1", _i),
        ("film", _vp), ("film_stride", _i), ("film_off", _i), ("gamma", _vp), ("beta", _vp), ("eps", _f),
        ("dst0", _vp), ("dst1", _vp), ("dst_raw0", _vp), ("dst_raw1", _vp),
        ("dst_lo0", _vp), ("dst_lo1", _vp), ("dst_raw_lo0", _vp), ("dst_raw_lo1", _vp),
    ]


class ConvDesc(C.Structure):
    _fields_ = [
        ("src0", _vp), ("src1", _vp), ("C0", _i), ("C1", _i), ("B", _i), ("H", _i), ("W", _i), ("taps", _i), ("stride", _i),
        ("wpk", _vp), ("bias", _vp), ("Cout", _i), ("CoutPad", _i),
        ("residual", _vp), ("out", _vp), ("out_stats", _vp), ("out_gs", _i), ("debug", _i), ("debug_buf", _vp),
        ("precise", _i), ("wpk_layout", _i), ("src0_lo", _vp), ("src1_lo", _vp),
        ("xsrc0", _vp), ("xsrc1", _vp), ("xsrc0_lo", _vp), ("xsrc1_lo", _vp), ("xC0", _i), ("xC1", _i), ("wpk_x", _vp), ("bias_x", _vp),
    ]


class DenoiserConfigC(C.Structure):
    _fields_ = [
        ("img_channels", _i), ("num_steps_conditioning", _i), ("cond_channels", _i), ("num_levels", _i),
        ("depths", _i * DMD_MAX_LEVELS), ("channels", _i * DMD_MAX_LEVELS), ("attn_depths", _i * DMD_MAX_LEVELS),
        ("num_actions", _i), ("sigma_data", _f), ("sigma_offset_noise", _f),
    ]


class ActorCriticConfigC(C.Structure):
    _fields_ = [
        ("lstm_dim", _i), ("img_channels", _i), ("img_size", _i), ("num_levels", _i),
        ("channels", _i * DMD_MAX_LEVELS), ("down", _i * DMD_MAX_LEVELS), ("num_actions", _i),
    ]


class RewEndConfigC(C.Structure):
    _fields_ = [
        ("lstm_dim", _i), ("img_channels", _i), ("img_size", _i), ("cond_channels", _i), ("num_levels", _i),
        ("depths", _i * DMD_MAX_LEVELS), ("channels", _i * DMD_MAX_LEVELS), ("attn_depths", _i * DMD_MAX_LEVELS), ("num_actions", _i),
    ]


class SamplerConfigC(C.Structure):
    _fields_ = [
        ("num_sigmas", _i), ("sigmas_host", C.POINTER(_f)), ("order", _i),
        ("s_churn", _f), ("s_tmin", _f), ("s_tmax", _f), ("s_noise", _f),
    ]


class WgradDesc(C.Structure):  # dmd_wgrad_desc
    _fields_ = [("grad", _vp), ("act", _vp), ("Cg", _i), ("Ca", _i), ("B", _i), ("H", _i), ("W", _i), ("taps", _i),
                ("dW", _vp), ("Cout", _i), ("Cin", _i), ("CinTot", _i), ("ci_off", _i), ("inv_scale", _vp),
                ("accumulate", _i), ("partial", _vp), ("partial_bytes", _sz), ("debug", _i)]


class ConvPlanInfo(C.Structure):  # dmd_conv_plan_info
    _fields_ = [("tiles", _i), ("kslabs", _i), ("stages", _i), ("tmem_cols", _i),
                ("smem_bytes", C.c_ulonglong), ("weight_bytes", C.c_ulonglong)]


# name -> (restype, argtypes); this table is also what tests use to check that every symbol is exported
SIGNATURES = {
    "dmd_version": (_i, []),
    "dmd_last_error": (C.c_char_p, []),
    "dmd_launch_count": (C.c_longlong, [_i]),
    "dmd_ktrace_begin": (_i, [_i]),
    "dmd_ktrace_end": (_i, [_vp, _i]),
    "dmd_ktrace_name": (C.c_char_p, [_i]),
    "dmd_pack_conv_weight": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "dmd_plc16_bytes": (_sz, [_i, _i, _i, _i]),
    "dmd_prep_act": (_i, [C.POINTER(PrepDesc), _vp]),
    "dmd_prep_plan": (_i, [C.POINTER(PrepDesc), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "dmd_conv_plan": (_i, [C.POINTER(ConvDesc), C.POINTER(ConvPlanInfo)]),
    "dmd_conv2d_fprop": (_i, [C.POINTER(ConvDesc), _vp]),
    "dmd_pack_conv_weight_dgrad": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
    "dmd_wgrad_partial_bytes": (_sz, []),
    "dmd_conv2d_wgrad": (_i, [C.POINTER(WgradDesc), _vp]),
    "dmd_gn_stats": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "dmd_attn_fwd": (_i, [_vp] * 10 + [_i, _i, _i, _i, _f, _vp]),
    "dmd_nchw_to_nhwc": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "dmd_nhwc_to_nchw": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "dmd_denoiser_create": (_vp, [C.POINTER(DenoiserConfigC)]),
    "dmd_denoiser_destroy": (None, [_vp]),
    "dmd_denoiser_num_tensors": (_i, [_vp]),
    "dmd_denoiser_packed_bytes": (_sz, [_vp]),
    "dmd_denoiser_set_weights": (_i, [_vp, C.POINTER(_vp), _i, _vp, _vp]),
    "dmd_denoiser_workspace_bytes": (_sz, [_vp, _i, _i, _i]),
    "dmd_denoiser_forward": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dmd_inner_model_forward": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dmd_denoiser_train_workspace_bytes": (_sz, [_vp, _i, _i, _i]),
    "dmd_denoiser_grad_layout": (C.c_longlong, [_vp, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong), _i]),
    "dmd_inner_model_forward_train": (_i, [_vp, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dmd_denoiser_backward": (_i, [_vp, _i, _i, _i, _vp, _vp, C.c_longlong, _vp, _vp]),
    "dmd_sampler_sample": (_i, [_vp, C.POINTER(SamplerConfigC), _i, _i, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _sz, _i, _vp]),
    "dmd_actor_critic_create": (_vp, [C.POINTER(ActorCriticConfigC)]),
    "dmd_actor_critic_destroy": (None, [_vp]),
    "dmd_actor_critic_num_tensors": (_i, [_vp]),
    "dmd_actor_critic_packed_bytes": (_sz, [_vp]),
    "dmd_actor_critic_set_weights": (_i, [_vp, C.POINTER(_vp), _i, _vp, _vp]),
    "dmd_actor_critic_workspace_bytes": (_sz, [_vp, _i]),
    "dmd_actor_critic_forward": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dmd_actor_critic_backward_scratch_bytes": (_sz, [_vp, _i]),
    "dmd_actor_critic_grad_layout": (C.c_longlong, [_vp, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong), _i]),
    "dmd_actor_critic_backward": (_i, [_vp, _i] + [_vp] * 8 + [C.c_longlong, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dmd_actor_critic_backward_accumulate": (_i, [_vp, _i] + [_vp] * 8 + [C.c_longlong, _vp, _vp, _vp, _vp, _sz, _vp]),
    "dmd_rew_end_create": (_vp, [C.POINTER(RewEndConfigC)]),
    "dmd_rew_end_destroy": (None, [_vp]),
    "dmd_rew_end_num_tensors": (_i, [_vp]),
    "dmd_rew_end_packed_bytes": (_sz, [_vp]),
    "dmd_rew_end_set_weights": (_i, [_vp, C.POINTER(_vp), _i, _vp, _vp]),
    "dmd_rew_end_workspace_bytes": (_sz, [_vp, _i]),
    "dmd_rew_end_predict": (_i, [_vp, _i, _i] + [_vp] * 9 + [_vp, _sz, _vp]),
    "dmd_rew_end_train_workspace_bytes": (_sz, [_vp, _i, _i]),
    "dmd_rew_end_grad_layout": (C.c_longlong, [_vp, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong), _i]),
    "dmd_rew_end_forward_train": (_i, [_vp, _i, _i] + [_vp] * 5 + [_vp, _sz, _vp]),
    "dmd_rew_end_backward": (_i, [_vp, _i, _i, _vp, _vp, _vp, C.c_longlong, _vp, _vp]),
    "dmd_lambda_returns": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, C.c_double, C.c_double, _vp]),
}

_lib: Optional[C.CDLL] = None


class LibraryMissing(RuntimeError):
    pass


def lib() -> C.CDLL:
    """Loads the native library; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LibraryMissing(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(diamond_b200 has no CPU / eager fallback)"
            )
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise RuntimeError("diamond_b200: " + lib().dmd_last_error().decode("utf-8", "replace"))


def ptr(t) -> Optional[int]:
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def current_stream() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream
