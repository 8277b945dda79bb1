"""ctypes binding of libc2w_b200.so (include/c2w_b200.h).  There is no CPU fallback: if the CUDA library is
missing or a call fails, this raises."""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

# C2W_LIB selects another build of the same ABI (tools/: the -DC2W_DIAG library with K1's cycle counters)
LIB_PATH = Path(os.environ.get("C2W_LIB") or Path(__file__).resolve().parent / "libc2w_b200.so")
MAX_LEVELS = 8
WS_VJP, WS_PER_SAMPLE_T, WS_TRAIN = 1, 2, 4


class C2WError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [
        ("frame_channels", C.c_int32),
        ("window", C.c_int32),
        ("height", C.c_int32),
        ("width", C.c_int32),
        ("embedding_dim", C.c_int32),
        ("noise_features", C.c_int32),
        ("n_levels", C.c_int32),
        ("hidden_channels", C.c_int32 * MAX_LEVELS),
        ("hidden_blocks", C.c_int32 * MAX_LEVELS),
        ("attention_mask", C.c_int32),
        ("forcing_dim", C.c_int32),
    ]


class AdamW(C.Structure):
    """include/c2w_b200.h: c2w_adamw"""
    _fields_ = [("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float),
                ("weight_decay", C.c_float), ("ema_rate", C.c_float), ("grad_scale", C.c_float), ("step", C.c_int32)]


class Guide(C.Structure):
    _fields_ = [
        ("x", C.c_void_p),
        ("eps", C.c_void_p),
        ("eps_out", C.c_void_p),
        ("y", C.c_void_p),
        ("std2", C.c_float * 8),   # C2W_MAX_VARS
        ("gamma", C.c_float * 8),
        ("mu", C.c_float),
        ("sigma", C.c_float),
        ("mu_next", C.c_float),
        ("sigma_next", C.c_float),
        ("t_step", C.c_int32),
        ("s_step", C.c_int32),
        ("H", C.c_int32),
        ("W", C.c_int32),
        ("frame_global0", C.c_int32),
        ("own_lo", C.c_int32),
        ("own_n", C.c_int32),
        ("mode", C.c_int32),
        ("partials", C.c_void_p),
        ("nan_flag", C.c_void_p),
        ("vjp", C.c_void_p),
        ("cot_out", C.c_void_p),
        ("halo", C.c_void_p),
        ("halo_k", C.c_int32),
        ("channels", C.c_int32),
    ]


class PointObs(C.Structure):
    """include/c2w_b200.h: c2w_point_obs"""
    _fields_ = [("frame_slot", C.c_void_p), ("strip_off", C.c_void_p), ("pix", C.c_void_p), ("ysum", C.c_void_p),
                ("wsum", C.c_void_p), ("n_slots", C.c_int32), ("strip_rows", C.c_int32)]


class ConvDesc(C.Structure):
    _fields_ = [
        ("x", C.c_void_p),
        ("n_img", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
        ("cin", C.c_int32),
        ("stride", C.c_int32),
        ("conv3x3", C.c_int32),
        ("w_packed", C.c_void_p),
        ("cout_pad", C.c_int32),
        ("bias", C.c_void_p),
        ("mode", C.c_int32),
        ("res", C.c_void_p),
        ("out", C.c_void_p),
        ("out_f32", C.c_void_p),
        ("bn", C.c_int32),
        ("variant", C.c_int32),
        ("max_ctas", C.c_int32),
        ("skip_loads", C.c_int32),
        ("ln_out", C.c_void_p),
        ("ln_mod", C.c_void_p),
        ("ln_upsample", C.c_int32),
        ("stats", C.c_void_p),
    ]


_vp, _i, _i64, _f, _d = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double

# name -> (restype, argtypes); every symbol include/c2w_b200.h declares
SIGNATURES = {
    "c2w_create": (_i, [C.POINTER(Config), C.POINTER(_vp)]),
    "c2w_destroy": (None, [_vp]),
    "c2w_last_error": (C.c_char_p, []),
    "c2w_abi_version": (_i, []),
    "c2w_struct_size": (_i, [_i]),
    "c2w_load_weight": (_i, [_vp, C.c_char_p, _vp, _i64]),
    "c2w_finalize_weights": (_i, [_vp]),
    "c2w_workspace_bytes": (_i64, [_vp, C.c_int32]),
    "c2w_bind_workspace": (_i, [_vp, C.c_int32, _vp, _i64]),
    "c2w_workspace_bytes_ex": (_i64, [_vp, C.c_int32, C.c_int32]),
    "c2w_bind_workspace_ex": (_i, [_vp, C.c_int32, _vp, _i64, C.c_int32]),
    "c2w_unet_forward_t": (_i, [_vp, _vp, C.c_int32, _vp, _vp, _vp]),
    "c2w_workspace_bytes_vjp": (_i64, [_vp, C.c_int32]),
    "c2w_bind_workspace_vjp": (_i, [_vp, C.c_int32, _vp, _i64]),
    "c2w_unet_vjp": (_i, [_vp, _vp, C.c_int32, _f, _vp, _vp, _vp, _vp]),
    "c2w_window_score_backward": (_i, [_vp, _vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _vp, _vp]),
    "c2w_window_score_sel": (_i, [_vp, _vp, C.c_int32, C.c_int32, _vp, C.c_int32, C.c_int32, _f, _vp, _vp]),
    "c2w_window_score_backward_sel": (_i, [_vp, _vp, C.c_int32, C.c_int32, _vp, _vp, C.c_int32, C.c_int32, _vp, _vp]),
    "c2w_unet_forward": (_i, [_vp, _vp, C.c_int32, _f, _vp, _vp]),
    "c2w_window_score": (_i, [_vp, _vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _f, _vp, _vp]),
    "c2w_traj_pack": (_i, [_vp, _vp, _i64, C.c_int32, C.c_int32, _vp]),
    "c2w_traj_unpack": (_i, [_vp, _vp, _i64, C.c_int32, C.c_int32, _vp]),
    "c2w_adamw_ema_step": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, C.POINTER(AdamW), _vp]),
    "c2w_normalize_pack": (_i, [_vp, _vp, _i64, C.c_int32, C.c_int32, C.c_int32, _vp, _vp, C.c_int32, _vp]),
    "c2w_unpack_unnormalize": (_i, [_vp, _vp, _i64, C.c_int32, C.c_int32, C.c_int32, _vp, _vp, C.c_int32, _vp]),
    "c2w_guided_step": (_i, [C.POINTER(Guide), _vp]),
    "c2w_guided_step_points": (_i, [C.POINTER(Guide), C.POINTER(PointObs), _vp]),
    "c2w_guided_step_combined": (_i, [C.POINTER(Guide), C.POINTER(PointObs), C.POINTER(C.c_float), _vp]),
    "c2w_guided_step_obs_std": (_i, [C.POINTER(Guide), C.POINTER(PointObs), _vp, _vp, _vp]),
    "c2w_reduce_partials": (_i, [_vp, C.c_int32, _vp, _vp]),
    "c2w_corrector_update": (_i, [_vp, _vp, _vp, _vp, _d, _f, _f, _i64, _i64, C.c_uint64, C.c_uint32, _vp, _vp]),
    "c2w_corrector_update_c": (_i, [_vp, _vp, _vp, _vp, _d, _f, _f, _i64, _i64, C.c_int32, C.c_uint64, C.c_uint32, _vp,
                                    _vp]),
    "c2w_op_conv_ex": (_i, [C.POINTER(ConvDesc), _vp]),
    "c2w_conv_tile_width": (_i, [_i, _i, _i, _i, _i, _i, _i]),
    "c2w_op_wgrad": (_i, [_vp, _vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _vp, _i64,
                          _vp, _vp, C.c_int32, C.c_int32, C.c_int32, _vp]),
    "c2w_op_colsum": (_i, [_vp, _vp, _i64, C.c_int32, _i64, C.c_int32, _f, _vp]),
    "c2w_op_conv": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "c2w_op_layernorm": (_i, [_vp, _vp, _vp, _i64, _i, _i, _i, _i, _vp]),
    "c2w_op_attention": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "c2w_op_layernorm_inv": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _vp]),
    "c2w_op_layernorm_bwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _i, _i, _i, _i, _vp]),
    "c2w_op_attention_bwd": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "c2w_op_gather_windows": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "c2w_op_modulation": (_i, [_vp, _f, _vp, _vp, _vp]),
    "c2w_total_mod_channels": (_i, [_vp]),
    "c2w_set_forcing": (_i, [_vp, _vp]),
    "c2w_param_total": (_i64, [_vp]),
    "c2w_refresh_weights": (_i, [_vp, _vp, _vp]),
    "c2w_param_layout": (_i, [_vp, C.c_char_p, C.POINTER(_i64), C.POINTER(_i64)]),
    "c2w_train_forward": (_i, [_vp, _vp, C.c_int32, _vp, _vp, _vp]),
    "c2w_train_backward": (_i, [_vp, _vp, C.c_int32, _vp, _vp, C.c_int32, _vp]),
    "c2w_dsm_loss_grad": (_i, [_vp, _vp, _vp, _i64, _f, _vp, _vp, _vp]),
    "c2w_train_step": (_i, [_vp, _vp, C.c_int32, _vp, _vp, _vp, _vp, _f, _vp, C.c_int32, _vp, _vp]),
    "c2w_halo_create": (_i, [_i64, C.POINTER(_vp)]),
    "c2w_halo_destroy": (None, [_vp]),
    "c2w_halo_handle": (_i, [_vp, _vp]),
    "c2w_halo_connect": (_i, [_vp, _vp, _vp]),
    "c2w_halo_exchange": (_i, [_vp, _vp, _i64, _i64, C.c_int32, _vp]),
    "c2w_halo_pull": (_i, [_vp, _vp, _i64, _i64, C.c_int32, _vp]),
    "c2w_halo_push_targets": (_i, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp),
                                   C.POINTER(C.c_uint32)]),
    "c2w_launch_count": (_i64, []),
    "c2w_set_timeline": (_i, [_vp, _vp, _i]),
    "c2w_set_timing": (_i, [_vp, _i]),
    "c2w_timing_read": (_i, [_vp, _vp, _vp]),
}

_lib = None


def load():
    """Loads the shared library (once).  Raises C2WError with the build recipe if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise C2WError(
            f"{LIB_PATH} not found: the CUDA extension is required (no CPU fallback). Build it with "
            "`python -m climate2weather_b200.build` or `python -c 'import __graft_entry__ as g; g.build()'`.")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().c2w_last_error()
        raise C2WError(f"{what} failed (rc={rc}): {msg.decode() if msg else '?'}")
