"""
ctypes binding of libtimbretrap_b200.so (include/timbre_trap_b200.h).

There is deliberately no fallback: if the shared library is missing or a call fails, an
exception is raised.  Build it with `python -c "import __graft_entry__ as g; g.build()"`
(or `python -m timbre_trap_b200.build`).
"""

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('TT_LIB_PATH') or os.path.join(_HERE, 'libtimbretrap_b200.so')   # override: A/B builds while tuning

_lib = None

c_void_p, c_int, c_int64, c_float_p, c_int32_p = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                                 ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_int32))

# name -> (restype, argtypes); every symbol include/timbre_trap_b200.h declares
SIGNATURES = {
    'tt_last_error': (ctypes.c_char_p, []),
    'tt_version': (c_int, []),
    'tt_launch_count': (ctypes.c_longlong, [c_int]),
    'tt_cqt_plan_create': (c_int, [ctypes.POINTER(c_void_p), c_int, c_int, c_int, c_int32_p, c_int32_p, c_int32_p,
                                   c_int32_p, c_float_p, c_float_p, c_int, c_int]),
    'tt_cqt_plan_destroy': (c_int, [c_void_p]),
    'tt_cqt_plan_set_lanes': (c_int, [c_void_p, c_int]),
    'tt_cqt_plan_scratch_bytes': (c_int64, [c_void_p]),
    'tt_cqt_forward': (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    'tt_cqt_inverse': (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p]),
    'tt_scale_by_peak': (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    'tt_magnitude': (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    'tt_chunk_crossfade': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    'tt_res_block_rs': (c_int, [c_void_p] * 5 + [c_int] * 7 + [c_void_p]),
    'tt_res_block_rs_mid': (c_int, [c_void_p] * 6 + [c_int] * 7 + [c_void_p]),
    'tt_set_strip_rows': (c_int, [c_int]),
    'tt_conv_down_strip': (c_int, [c_void_p] * 3 + [c_int] * 7 + [c_void_p]),
    'tt_conv_up_strip': (c_int, [c_void_p] * 3 + [c_int] * 8 + [c_void_p]),
    'tt_conv_same': (c_int, [c_void_p] * 4 + [c_int] * 7 + [c_void_p]),
    'tt_conv_same_post': (c_int, [c_void_p] * 4 + [c_int] * 8 + [c_void_p] * 2),
    'tt_conv_lat': (c_int, [c_void_p] * 4 + [c_int] * 5 + [c_void_p]),
    'tt_deconv_in': (c_int, [c_void_p] * 4 + [c_int] * 6 + [c_void_p]),
    'tt_conv_in': (c_int, [c_void_p] * 4 + [c_int] * 5 + [c_void_p]),
    'tt_conv_out': (c_int, [c_void_p] * 4 + [c_int] * 5 + [c_void_p]),
    'tt_conv_out_crossfade': (c_int, [c_void_p] * 4 + [c_int] * 5 + [c_void_p] * 3),
    'tt_cqt_inverse_clips': (c_int, [c_void_p] * 3 + [c_int] * 2 + [c_void_p] * 2 + [c_int, c_void_p]),
    'tt_scale_by_clip_peak': (c_int, [c_void_p] * 2 + [c_int] * 3 + [c_void_p] * 2),
    'tt_gather_chunks': (c_int, [c_void_p] * 2 + [c_int] * 4 + [c_void_p] * 2),
    'tt_chunk_crossfade_clips': (c_int, [c_void_p] * 3 + [c_int] * 4 + [c_void_p] * 3),
    'tt_conv_out_crossfade_clips': (c_int, [c_void_p] * 5 + [c_int] * 6 + [c_void_p] * 3),
    'tt_add_scaled_bf16': (c_int, [c_void_p] * 4 + [c_int64, c_void_p]),
    'tt_dot_scratch_floats': (c_int, []),
    'tt_dot_bf16': (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    'tt_widen_pairs': (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    'tt_pairs_to_c8': (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    'tt_channel0_activation': (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    'tt_channel0_activation_bwd': (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    'tt_resample_mono': (c_int, [c_void_p, c_int, c_int64, c_void_p, c_int, c_int, c_int, c_void_p, c_int64, c_void_p, c_void_p]),
    'tt_rasterise_pitches': (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    'tt_sdr_correlations': (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    'tt_loss_scratch_floats': (c_int, []),
    'tt_sum_sq_diff': (c_int, [c_void_p, c_void_p, c_int64, ctypes.c_double, c_void_p, c_void_p, c_void_p]),
    'tt_transcription_loss': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    'tt_wgrad_scratch_floats': (c_int64, [c_int, c_int, c_int]),
    'tt_conv_wgrad_same': (c_int, [c_void_p] * 4 + [c_int] * 9 + [c_void_p, c_void_p]),
    'tt_conv_wgrad_updown': (c_int, [c_void_p] * 4 + [c_int] * 9 + [c_void_p, c_void_p]),
    'tt_wgrad_lat_scratch_floats': (c_int64, [c_int, c_int, c_int]),
    'tt_conv_wgrad_lat': (c_int, [c_void_p] * 5 + [c_int] * 7 + [c_void_p, c_void_p]),
    'tt_elu_bwd_bf16': (c_int, [c_void_p] * 3 + [c_int64, c_void_p]),
    'tt_res_out_bwd_bf16': (c_int, [c_void_p] * 4 + [c_int64, c_void_p]),
    'tt_p4_to_c8': (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    'tt_c8_to_p4': (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    'tt_sum_sq_diff_bwd': (c_int, [c_void_p] * 3 + [ctypes.c_double] + [c_void_p] * 2 + [c_int64, c_void_p]),
    'tt_transcription_loss_bwd': (c_int, [c_void_p] * 3 + [c_int] * 4 + [c_void_p] * 3),
    'tt_activations_bwd': (c_int, [c_void_p] * 3 + [c_int64, c_void_p]),
    'tt_film_convin_grad': (c_int, [c_void_p] * 7 + [c_int] * 4 + [c_void_p] * 7),
    'tt_grad_sumsq': (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    'tt_adamw_step': (c_int, [c_void_p] * 4 + [c_int64, c_void_p] + [ctypes.c_float] * 6 + [c_int, c_void_p]),
    'tt_to_decibels': (c_int, [c_void_p, c_int, c_int64, c_int, c_void_p, c_void_p, c_void_p]),
    'tt_filter_non_peaks': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    'tt_peak_threshold': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, ctypes.c_float, c_int, c_int, c_int, c_void_p]),
    'tt_multipitch_counts': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
}


class TimbreTrapB200Error(RuntimeError):
    pass


def lib():
    """The loaded shared library (loads on first use; raises if it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise TimbreTrapB200Error(
                f'{LIB_PATH} is missing - the CUDA extension has not been built (run __graft_entry__.build()). '
                'timbre_trap_b200 has no CPU or PyTorch fallback.')
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)      # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(status):
    if status != 0:
        msg = lib().tt_last_error()
        raise TimbreTrapB200Error(f'timbre_trap_b200 call failed (status {status}): {msg.decode() if msg else "?"}')


def require_cuda(tensor, what):
    if not tensor.is_cuda:
        raise TimbreTrapB200Error(f'{what} must be a CUDA tensor: timbre_trap_b200 has no CPU path '
                                  '(the CPU oracle lives in oracle/ and is test-only).')
