"""ctypes binding of libcomet_b200.so (the C ABI declared in include/comet_b200.h).

There is deliberately no fallback: if the shared library has not been built (``python -m
comet_pose_estimation_b200.build`` or ``__graft_entry__.build()``) importing this module raises, and every
compute call on a machine without a CUDA device fails with the library's own error."""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libcomet_b200.so")

OK, ERR_INVALID, ERR_CUDA, ERR_UNSUPPORTED = 0, 1, 2, 3
PAD_ZEROS, PAD_BORDER = 0, 1
PREC_F32, PREC_BF16_AUTOCAST = 0, 1
PYR_NCHW, PYR_CHANNEL_LAST, PYR_ALL_CHANNEL_LAST, PYR_UP2_SOURCE = 0, 1, 2, 3
FMAPS_NCHW, FMAPS_CHANNEL_LAST = 0, 1
MAX_LEVELS, MAX_RADIUS = 8, 7
OPT_TENSOR_PATH, OPT_TMA_LOOKUP, OPT_GEMM_BK32, OPT_TC_OVERLAP_MISC, OPT_TC_REDUCE_STORE, OPT_GEMM_TMA_STORE, OPT_GEMM_EW16, OPT_GEMM_BN96, OPT_GEMM_PAIR, OPT_ATTN_MMA = 0, 1, 2, 3, 4, 5, 6, 7, 8, 9

_p = C.c_void_p
_i = C.c_int
_ll = C.c_longlong

# name -> (restype, argtypes); mirrors include/comet_b200.h one to one (tests/test_cabi.py checks that).
SIGNATURES = {
    "comet_version": (_i, []),
    "comet_last_error": (C.c_char_p, []),
    "comet_has_tensor_path": (_i, []),
    "comet_launch_count": (_ll, []),
    "comet_pyramid_offset": (_ll, [_i, _i, _i, _i, _i]),
    "comet_pyramid_elems": (_ll, [_i, _i, _i, _i, _i]),
    "comet_pyramid_f32": (_i, [_p, _p, _i, _i, _i, _i, _i, _p]),
    "comet_corr_volume_f32": (_i, [_p, _ll, _ll, _p, _p, _i, _i, _i, _i, _i, _p]),
    "comet_pyramid_cl_f32": (_i, [_p, _p, _i, _i, _i, _i, _i, _i, _p]),
    "comet_pyramid_up2_elems": (_ll, [_i, _i, _i, _i]),
    "comet_pyramid_up2_f32": (_i, [_p, _p, _i, _i, _i, _i, _p]),
    "comet_up2_supported": (_i, [_i, _i, _i, _i, _i, _i]),
    "comet_corr_lookup_f32": (_i, [_p, _p, _p, _ll, _ll, _ll, _i, _p, _ll, _ll, _ll, _p, _ll, _ll, _ll,
                                   _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p]),
    "comet_track_tokens_f32": (_i, [_p, _p, _p, _ll, _ll, _ll, _p, _ll, _ll, _ll, _p, _p,
                                    _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p]),
    "comet_track_tokens_ragged_f32": (_i, [_p, _p, _p, _ll, _ll, _ll, _p, _ll, _ll, _ll, _p, _p, _p,
                                           _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p]),
    "comet_track_tokens_varlen_f32": (_i, [_p, _p, _p, _ll, _ll, _ll, _p, _ll, _ll, _ll, _p, _p, _p, _p,
                                           _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p]),
    "comet_track_tokens_indexed_f32": (_i, [_p, _p, _p, _ll, _ll, _ll, _p, _ll, _ll, _ll, _p, _p, _p, _p, _p, _i,
                                            _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p]),
    "comet_sampled_pos_emb_f32": (_i, [_p, _ll, _ll, _p, _i, _i, _i, _i, _i, _p]),
    "comet_bilinear_sampler4d_f32": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _p]),
    "comet_bilinear_sampler5d_f32": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p]),
    "comet_sample_features4d_f32": (_i, [_p, _ll, _p, _ll, _ll, _p, _i, _i, _i, _i, _i, _p]),
    "comet_sample_features4d_cl_f32": (_i, [_p, _ll, _p, _ll, _ll, _p, _i, _i, _i, _i, _i, _p]),
    "comet_upsample_bilinear_ac_f32": (_i, [_p, _p, _ll, _i, _i, _i, _i, _i, _i, _p]),
    "comet_upsample_bilinear_ac_bf16": (_i, [_p, _p, _ll, _i, _i, _i, _i, _i, _p]),
    "comet_instance_norm_f32": (_i, [_p, _p, _ll, _i, _i, _i, _i, C.c_float, _p]),
    "comet_instance_norm_bf16": (_i, [_p, _p, _ll, _i, _i, _i, C.c_float, _p]),
    "comet_extract_patches_f32": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p]),
    "comet_shallow_encoder_packed_elems": (_ll, []),
    "comet_shallow_encoder_pack_f32": (_i, [_p, _p, _p]),
    "comet_shallow_encoder_f32": (_i, [_p, _ll, _ll, _ll, _ll, _p, _p, _ll, C.c_float, _p]),
    "comet_shallow_encoder_from_images_f32": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, C.c_float, _p]),
    "comet_shallow_encoder_from_images_ragged_f32": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, C.c_float, _p]),
    "comet_shallow_encoder_from_images_varlen_f32": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, C.c_float, _p]),
    "comet_shallow_encoder_from_images_indexed_f32": (_i, [_p, _p, _p, _p, _p, _i, _p, _p, _i, _i, _i, _i, _i, C.c_float,
                                                           _p]),
    "comet_shallow_encoder_from_images_packed_f32": (_i, [_p, _p, _p, _ll, _p, _p, _p, _p, _p, _p, _i, _i, _i, C.c_float,
                                                          _p]),
    "comet_embed2d_f32": (_i, [_p, _p, _ll, _i, _i, _p]),
    "comet_sincos1d_from_grid_f32": (_i, [_p, _p, _ll, _i, _p]),
    "comet_sincos2d_f32": (_i, [_p, _i, _i, _i, _p]),
    "comet_tc_supported": (_i, [_i, _i, _i, _i, _i, _i]),
    "comet_tc_split_elems": (_ll, [_i]),
    "comet_tc_workspace_bytes": (_ll, [_i, _i]),
    "comet_tc_prepare_f32": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _p]),
    "comet_tc_corr_lookup_f32": (_i, [_p, _p, _ll, _ll, _ll, _p, _ll, _ll, _ll, _p, _ll, _ll, _ll,
                                      _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p]),
    "comet_tc_track_tokens_f32": (_i, [_p, _p, _ll, _ll, _ll, _p, _ll, _ll, _ll, _p, _p,
                                       _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p]),
    "comet_tc_track_tokens_ragged_f32": (_i, [_p, _p, _ll, _ll, _ll, _p, _ll, _ll, _ll, _p, _p, _p,
                                              _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p]),
    "comet_tc_track_tokens_varlen_f32": (_i, [_p, _p, _ll, _ll, _ll, _p, _ll, _ll, _ll, _p, _p, _p, _p,
                                              _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p]),
    "comet_tc_track_tokens_indexed_f32": (_i, [_p, _p, _ll, _ll, _ll, _p, _ll, _ll, _ll, _p, _p, _p, _p, _p, _i,
                                               _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p]),
    "comet_tc_corr_volume_f32": (_i, [_p, _p, _ll, _ll, _ll, _p, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p]),
    "comet_tc_status": (_i, []),
    "comet_split_planes_f32": (_i, [_p, _ll, _p, _ll, _ll, _ll, _i, _i, _p]),
    "comet_linear_tc": (_i, [_p, _ll, _ll, _p, _ll, _ll, _i, _p, _p, _ll, _p, _ll, _p, _ll, _ll, _i, _i, _ll, _i, _i, _p]),
    "comet_layernorm_planes_f32": (_i, [_p, _ll, _p, _p, C.c_float, _p, _ll, _p, _ll, _ll, _i, _ll, _i, _p]),
    "comet_attention_planes_f32": (_i, [_p, _ll, _ll, _p, _ll, _ll, _p, _ll, _ll, _p, _ll, _ll, _ll, _i, _i, _i, _i, _i, _i, _p]),
    "comet_attention_varlen_planes_f32": (_i, [_p, _ll, _ll, _p, _ll, _ll, _p, _p, _ll, _ll, _i, _i, _i, _i,
                                               _p, _p, _p, _p, _i, _i, _i, _i, _i, _p]),
    "comet_attention_varlen_grouped_planes_f32": (_i, [_p, _ll, _ll, _p, _ll, _ll, _p, _p, _ll, _ll, _i, _i, _i, _i,
                                                       _p, _p, _p, _p, _i, _i, _i, _i, _p, _i, _i, _p]),
    "comet_add_planes_f32": (_i, [_p, _p, _p, _ll, _i, _ll, _p]),
    "comet_set_option": (_i, [_i, _i]),
    "comet_get_option": (_i, [_i]),
}


class CometB200Error(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build the sm_100a kernels first (python -m comet_pose_estimation_b200.build). "
            "comet_pose_estimation_b200 has no CPU or PyTorch fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the ABI and this table disagree
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def set_option(option: int, value: bool) -> bool:
    """Library-wide A/B switch (``OPT_TENSOR_PATH``, ``OPT_TMA_LOOKUP``); returns the previous value."""
    prev = bool(lib.comet_get_option(option))
    check(lib.comet_set_option(option, int(bool(value))))
    return prev


def last_error() -> str:
    return (lib.comet_last_error() or b"").decode("utf-8", "replace")


def check(rc: int) -> None:
    """Map the C status to the exception the reference would raise for the same condition
    (its hot path only uses ``assert``, SURVEY.md 8b)."""
    if rc == OK:
        return
    msg = last_error()
    if rc == ERR_INVALID:
        raise AssertionError(msg)
    raise CometB200Error(f"comet_b200 error {rc}: {msg}")
