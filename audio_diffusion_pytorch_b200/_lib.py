"""ctypes binding of libadp_b200.so (C ABI declared in include/adp_b200.h).

There is deliberately no fallback: if the shared library is missing or the device is not
sm_100 the product path raises.  Nothing under oracle/ is imported here.
"""
import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libadp_b200.so")

i32, f32, vp = C.c_int32, C.c_float, C.c_void_p


class ConvGemmArgs(C.Structure):
    _fields_ = [("a", vp), ("w", vp), ("out", vp), ("bias", vp), ("residual", vp), ("gate", vp),
                ("stats", vp), ("B", i32), ("T", i32), ("c_in", i32), ("lda", i32), ("ldo", i32),
                ("k_total", i32), ("n_pad", i32), ("n_valid", i32), ("phases", i32),
                ("ntaps", i32), ("tap_off", i32 * 3), ("up_factor", i32), ("groups", i32),
                ("block_n", i32), ("out_fp32", i32), ("ld_gate", i32)]


class StemInArgs(C.Structure):
    _fields_ = [("x", vp), ("append", vp), ("noise", vp), ("alpha", vp), ("beta", vp), ("w", vp),
                ("bias", vp), ("out", vp), ("stats", vp), ("B", i32), ("T", i32), ("cx", i32),
                ("ca", i32), ("c0", i32), ("f", i32), ("groups", i32)]


class StemOutArgs(C.Structure):
    _fields_ = [("h", vp), ("x", vp), ("append", vp), ("w", vp), ("bias", vp), ("w_adapt", vp),
                ("b_adapt", vp), ("gate", vp), ("v_out", vp), ("x_next", vp), ("ab", vp),
                ("noise", vp), ("alpha", vp), ("beta", vp), ("loss_sum", vp), ("dv", vp),
                ("cfg_scale", f32), ("cfg", i32), ("B", i32), ("T", i32), ("cx", i32),
                ("ca", i32), ("c0", i32), ("co", i32), ("f", i32), ("ld_gate", i32)]


class NarrowConvArgs(C.Structure):
    _fields_ = [("x", vp), ("y", vp), ("stats_in", vp), ("gamma", vp), ("beta", vp), ("w", vp),
                ("bias", vp), ("residual", vp), ("scale_shift", vp), ("stats_out", vp),
                ("ss_stride", i32), ("B", i32), ("T", i32), ("C", i32), ("groups", i32),
                ("gn_eps", f32), ("ln_eps", f32), ("w_packed", vp)]


class WgradArgs(C.Structure):
    _fields_ = [("g", vp), ("x", vp), ("dw", vp), ("B", i32), ("T", i32), ("n", i32), ("k", i32),
                ("ldg", i32), ("ldx", i32), ("ldw", i32), ("g_cols", i32), ("x_cols", i32),
                ("g_col0", i32), ("x_col0", i32), ("off", i32), ("ntaps", i32),
                ("tap_stride", C.c_int64)]


class NarrowConvBwdArgs(C.Structure):
    _fields_ = [("dy", vp), ("x", vp), ("stats_in", vp), ("gamma", vp), ("beta", vp), ("w", vp),
                ("dxh", vp), ("dgamma", vp), ("dbeta", vp), ("S", vp), ("dw", vp), ("dbias", vp),
                ("B", i32), ("T", i32), ("C", i32), ("groups", i32), ("gn_eps", f32)]


class StemOutBwdArgs(C.Structure):
    _fields_ = [("dv", vp), ("gscale", vp), ("h", vp), ("x", vp), ("append", vp), ("noise", vp),
                ("alpha", vp), ("beta", vp), ("w", vp), ("bias", vp), ("w_adapt", vp), ("gate", vp),
                ("dh", vp), ("dw", vp), ("dbias", vp), ("dgate", vp), ("dw_adapt", vp),
                ("db_adapt", vp), ("dxin", vp), ("B", i32), ("T", i32), ("cx", i32), ("ca", i32), ("c0", i32),
                ("co", i32), ("f", i32), ("ld_gate", i32), ("ld_dgate", i32)]


class StemInBwdArgs(C.Structure):
    _fields_ = [("dout", vp), ("x", vp), ("append", vp), ("noise", vp), ("alpha", vp), ("beta", vp),
                ("dw", vp), ("dbias", vp), ("w", vp), ("dxin", vp), ("B", i32), ("T", i32),
                ("cx", i32), ("ca", i32), ("c0", i32), ("f", i32)]


class AttentionBwdArgs(C.Structure):
    _fields_ = [("q", vp), ("k", vp), ("v", vp), ("o", vp), ("d_o", vp), ("lse", vp), ("delta", vp),
                ("dq", vp), ("dk", vp), ("dv", vp), ("B", i32), ("H", i32), ("Tq", i32), ("Tk", i32),
                ("ldq", i32), ("ldk", i32), ("ldv", i32), ("ldo", i32), ("lddo", i32), ("lddq", i32),
                ("lddk", i32), ("lddv", i32), ("scale", f32)]


_lib = None


def lib() -> C.CDLL:
    """Loads the library once.  Raises (never falls back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU / PyTorch fallback for the audio-diffusion hot path)")
    L = C.CDLL(LIB_PATH)
    L.adp_last_error.restype = C.c_char_p
    L.adp_version.restype = i32
    sig = {
        "adp_device_check": [],
        "adp_debug_set": [i32, i32],
        "adp_conv_gemm": [C.POINTER(ConvGemmArgs), vp],
        "adp_gn_silu": [vp, vp, vp, vp, vp, i32, i32, i32, i32, f32, vp],
        "adp_gn_stats": [vp, vp, i32, i32, i32, i32, vp],
        "adp_ln_film": [vp, vp, vp, i32, vp, i32, i32, i32, i32, f32, vp],
        "adp_ln_film_dual": [vp, vp, vp, vp, i32, vp, i32, i32, i32, i32, f32, f32, vp],
        "adp_attention": [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, f32, vp, vp],
        "adp_attention_bwd": [C.POINTER(AttentionBwdArgs), vp],
        "adp_ln_fold_bwd": [vp, vp, vp, vp, i32, vp, vp, vp, vp, i32, i32, vp],
        "adp_skinny_linear": [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp],
        "adp_time_features": [vp, vp, vp, i32, i32, i32, vp],
        "adp_stem_in": [C.POINTER(StemInArgs), vp],
        "adp_stem_out": [C.POINTER(StemOutArgs), vp],
        "adp_narrow_conv": [C.POINTER(NarrowConvArgs), vp],
        "adp_sampler_step": [vp, vp, vp, vp, C.c_int64, vp],
        "adp_inpaint_blend": [vp, vp, vp, vp, vp, C.c_int64, vp],
        "adp_arv_step": [vp, vp, vp, C.c_int, C.c_int, C.c_int, vp],
        "adp_resample": [vp, vp, vp] + [C.c_int] * 7 + [vp],
        "adp_resample_adjoint": [vp, vp, vp] + [C.c_int] * 7 + [vp],
        "adp_mel_spectrogram": [vp] * 5 + [C.c_int] * 8 + [vp],
        "adp_to_flat": [vp, vp, vp] + [C.c_int] * 7 + [vp],
        "adp_to_flat_bwd": [vp] * 5 + [C.c_int] * 7 + [vp],
        "adp_f32_conv_gemm": [C.POINTER(ConvGemmArgs), vp],
        "adp_f32_gn_stats": [vp, vp, i32, i32, i32, i32, vp],
        "adp_f32_gn_silu": [vp, vp, vp, vp, vp, i32, i32, i32, i32, f32, vp],
        "adp_f32_ln_film": [vp, vp, vp, vp, i32, i32, i32, i32, f32, f32, vp],
        "adp_f32_attention": [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, f32, vp],
        "adp_f32_linear": [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp],
        "adp_f32_silu": [vp, vp, C.c_int64, vp],
        "adp_f32_stem_in": [C.POINTER(StemInArgs), vp],
        "adp_f32_stem_out": [C.POINTER(StemOutArgs), vp],
        "adp_step_select": [vp, vp, vp, vp, vp, C.c_int64, vp],
        "adp_step_advance": [vp, vp],
        "adp_silu_bf16": [vp, vp, C.c_int64, vp],
        "adp_wgrad": [C.POINTER(WgradArgs), vp],
        "adp_gn_silu_bwd": [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, f32, vp],
        "adp_gn_bwd_apply": [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, f32, vp],
        "adp_ln_film_bwd": [vp, vp, vp, i32, vp, vp, i32, vp, vp, i32, i32, i32, f32, vp],
        "adp_colsum": [vp, vp, i32, vp, i32, i32, i32, vp],
        "adp_skip_gate": [vp, vp, vp, i32, vp, vp, i32, i32, i32, i32, vp],
        "adp_skip_gate_bwd": [vp, vp, vp, i32, vp, vp, i32, i32, i32, i32, vp],
        "adp_cond_bwd": [vp, i32, vp, vp, vp, vp, vp, i32, i32, i32, vp],
        "adp_narrow_conv_bwd": [C.POINTER(NarrowConvBwdArgs), vp],
        "adp_stem_out_bwd": [C.POINTER(StemOutBwdArgs), vp],
        "adp_stem_in_bwd": [C.POINTER(StemInBwdArgs), vp],
    }
    for name, argtypes in sig.items():
        if hasattr(L, name):
            fn = getattr(L, name)
            fn.argtypes = argtypes
            fn.restype = i32
    _lib = L
    return L


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"{what} failed: {lib().adp_last_error().decode()}")


EXPORTS = ["adp_version", "adp_last_error", "adp_device_check", "adp_conv_gemm", "adp_gn_silu",
           "adp_gn_stats", "adp_ln_film", "adp_ln_film_dual", "adp_attention", "adp_skinny_linear",
           "adp_time_features", "adp_stem_in", "adp_stem_out", "adp_narrow_conv",
           "adp_sampler_step", "adp_silu_bf16", "adp_debug_set", "adp_wgrad", "adp_gn_silu_bwd",
           "adp_gn_bwd_apply", "adp_ln_film_bwd", "adp_colsum", "adp_skip_gate",
           "adp_skip_gate_bwd", "adp_cond_bwd", "adp_narrow_conv_bwd", "adp_stem_out_bwd",
           "adp_stem_in_bwd", "adp_attention_bwd", "adp_ln_fold_bwd", "adp_inpaint_blend", "adp_arv_step", "adp_resample", "adp_resample_adjoint",
           "adp_mel_spectrogram", "adp_to_flat", "adp_to_flat_bwd", "adp_f32_conv_gemm", "adp_f32_gn_stats",
           "adp_f32_gn_silu", "adp_f32_ln_film", "adp_f32_attention", "adp_f32_linear", "adp_f32_silu",
           "adp_f32_stem_in", "adp_f32_stem_out", "adp_step_select", "adp_step_advance"]
