"""ctypes binding of libflowhigh_b200.so (the C ABI declared in include/flowhigh_b200.h).

No torch types cross this boundary: tensors are passed as raw device addresses
(`tensor.data_ptr()`), sizes as ints, the stream as a void*.  A missing library is a hard
error -- there is no CPU or PyTorch fallback for any kernel.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

from .build import lib_path

_i, _i64, _f, _p = C.c_int, C.c_int64, C.c_float, C.c_void_p


class TcConvArgs(C.Structure):
    """Mirror of `fh_tc_conv_args` (include/flowhigh_b200.h)."""
    _fields_ = [
        ("a", _p), ("a_batch", _i64), ("a_chunk", _i64), ("a_row0", _i),
        ("w", _p), ("bias", _p), ("res", _p), ("out", _p),
        ("out_batch", _i64), ("out_chunk", _i64), ("out_row", _i64),
        ("res_batch", _i64), ("res_chunk", _i64), ("res_row", _i64),
        ("out_is_16", _i), ("res_is_16", _i),
        ("alpha", _f), ("beta_res", _f),
        ("accumulate", _i), ("geglu", _i),
        ("B", _i), ("L", _i), ("Cin", _i), ("Cout", _i),
        ("ntaps", _i), ("P", _i),
        ("tap_off", C.POINTER(_i)),
        ("bn", _i),
        ("fp16", _i),
        ("act", _i),
        ("acc_src", _p),
        ("two_cta", _i),
    ]


# name -> (restype, argtypes); every symbol include/flowhigh_b200.h declares
SIGNATURES = {
    "fh_version": (_i, []),
    "fh_last_error_string": (C.c_char_p, []),
    "fh_launch_count": (_i64, []),
    "fh_set_status_word": (_i, [_p]),
    "fh_set_debug_word": (_i, [_p]),
    "fh_resample_poly_f32": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _p]),
    "fh_scale_by_absmax_f32": (_i, [_p, _p, _p, _f, _i, _i, _p]),
    "fh_absmax_f32": (_i, [_p, _p, _i, _i, _p]),
    "fh_fill_u32": (_i, [_p, C.c_uint32, _i64, _p]),
    "fh_stft_logmel_f32": (_i, [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p]),
    "fh_pp_cutoff": (_i, [_p, _p, _i, _f, _p]),
    "fh_pp_energy_ws_bytes": (_i, [_i, _i]),
    "fh_pp_src_energy_f32": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _p]),
    "fh_pp_fused_f32": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p]),
    "fh_pp_overlap_add_f32": (_i, [_p, _p, _p, _p, _i, _i, _i, _p]),
    "fh_ola_crossfade_f32": (_i, [_p, _p, _i, _i, _i, _i64, _p]),
    "fh_sgemm_nt_f32": (_i, [_p, _i, _p, _i, _p, _p, _i, _f, _f, _p, _i, _i, _i, _i, _p]),
    "fh_gemv_f32": (_i, [_p, _p, _p, _p, _i, _i, _i, _p]),
    "fh_sincos_embed_f32": (_i, [_p, _f, _p, _i, _p]),
    "fh_dwconv_gelu_res_f32": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _p]),
    "fh_dwconv_f32": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _p]),
    "fh_layernorm_f32": (_i, [_p, _p, _p, _p, _i, _i64, _i, _i, _f, _p]),
    "fh_gelu_f32": (_i, [_p, _p, _i, _i, _p]),
    "fh_rmsnorm_f32": (_i, [_p, _p, _p, _p, _i, _i64, _i, _i, _p]),
    "fh_qknorm_rope_f32": (_i, [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p]),
    "fh_attention_f32": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _f, _p]),
    "fh_attention_tc5_operand_elems": (_i64, [_i, _i, _i, _i]),
    "fh_qknorm_rope_tiles": (_i, [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _f, _i, _p]),
    "fh_attention_tc5": (_i, [_p, _p, _p, _p, _i, _i64, _i, _i, _i, _i, _i, _p]),
    "fh_geglu_f32": (_i, [_p, _p, _i, _i, _p]),
    "fh_axpby_f32": (_i, [_p, _p, _f, _f, _p, _i64, _p]),
    "fh_rk_lincomb_f32": (_i, [_p, _p, _i64, _i, C.POINTER(_f), _p, _i64, _p]),
    "fh_rk_scaled_sumsq_f32": (_i, [_p, _p, _p, _f, _f, _i, _i64, _p, _p]),
    "fh_broadcast_row_f32": (_i, [_p, _p, _i64, _i, _p]),
    "fh_mel_cutoff_f32": (_i, [_p, _p, _i, _i, _i, _f, _p]),
    "fh_mel_splice_f32": (_i, [_p, _p, _p, _p, _i, _i, _i, _p]),
    "fh_conv1d_taps_f32": (_i, [_p, _p, _p, _p, _p, _f, _f, _i, _p, _i, _i, _i, _i, _i, _i, _p]),
    "fh_snake_aa_f32": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _p]),
    "fh_convpost_tanh_f32": (_i, [_p, _p, _f, _p, _i, _i, _i, _p]),
    "fh_transpose_f32": (_i, [_p, _p, _i, _i, _i, _p]),
    "fh_cast_f32_16": (_i, [_p, _p, _i64, _i, _p]),
    "fh_cast_f32_16_split": (_i, [_p, _p, _i64, _i, _i64, _i64, _i, _i, _p]),
    "fh_sum_cast_f32": (_i, [_p, _p, _p, _p, _p, _p, _i64, _i, _p]),
    "fh_tc_conv": (_i, [C.POINTER(TcConvArgs), _p]),
    "fh_tc_packed_weight_bytes": (_i64, [_i, _i, _i, _i, _i]),
    "fh_to_chunked_16": (_i, [_p, _i64, _i64, _i64, _p, _i64, _i64, _i, _i, _i, _i, _i, _p]),
    "fh_to_chunked_16_split": (_i, [_p, _i64, _i64, _i64, _p, _i64, _i64, _i, _i, _i, _i, _i, _p]),
    "fh_snake_aa_chunked_split": (_i, [_p, _p, _p, _p, _p, _i64, _i64, _i64, _i, _i, _i, _i, _p]),
    "fh_snake_aa_chunked": (_i, [_p, _p, _p, _p, _p, _i64, _i64, _i, _i, _i, _i, _i, _p]),
    "fh_snake_aa_chunked_h": (_i, [_p, _p, _p, _p, _p, _i64, _i64, _i, _i, _i, _i, _p]),
    "fh_snakepost_convpost_tanh": (_i, [_p, _i64, _i64, _i, _p, _p, _p, _p, _f, _p, _i, _i, _i, _p]),
    "fh_convpost_tanh_chunked": (_i, [_p, _i64, _i64, _i, _p, _f, _p, _i, _i, _i, _p]),
}

_lib: Optional[C.CDLL] = None


class FlowHighNativeError(RuntimeError):
    pass


def load(build_if_missing: bool = True) -> C.CDLL:
    """Loads the shared library (building it in-tree first if the sources are newer)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if build_if_missing and os.environ.get("FLOWHIGH_B200_NO_BUILD") != "1":
        try:
            from .build import build
            path = build()
        except Exception as e:  # nvcc missing on a deployment box: the prebuilt .so must exist
            if not os.path.exists(path):
                raise FlowHighNativeError(f"libflowhigh_b200.so is missing and cannot be built: {e}") from e
    if not os.path.exists(path):
        raise FlowHighNativeError(
            f"{path} not found: run `python -m flowhigh_b200.build` (nvcc, sm_100a). There is no fallback path.")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().fh_last_error_string().decode("utf-8", "replace")
        exc = ValueError if rc in (-1, -2, -3) else FlowHighNativeError
        raise exc(f"{what or 'flowhigh_b200'} failed (rc={rc}): {msg}")


def call(name: str, *args) -> None:
    check(getattr(load(), name)(*args), name)


def launch_count() -> int:
    return int(load().fh_launch_count())
