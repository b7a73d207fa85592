"""ctypes binding of include/vadb200.h.  Fails loudly when the CUDA library is missing:
there is no CPU fallback anywhere in this package."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VADB200_LIB") or os.path.join(HERE, "libvadb200.so")  # override: A/B experiments only


class VadB200Error(RuntimeError):
    def __init__(self, code, msg):
        RuntimeError.__init__(self, "vadb200 error %d: %s" % (code, msg))
        self.code = code


class TreeFitParams(C.Structure):
    _fields_ = [("max_depth", C.c_int32), ("min_samples_split", C.c_int32), ("min_samples_leaf", C.c_int32),
                ("reserved", C.c_int32), ("min_impurity_decrease", C.c_double)]


class Config(C.Structure):
    _fields_ = [("sample_rate", C.c_int32), ("frame_size", C.c_int32), ("frame_step", C.c_int32),
                ("fft_n", C.c_int32), ("n_filters", C.c_int32), ("n_mfcc", C.c_int32),
                ("low_hz", C.c_double), ("high_hz", C.c_double), ("lifter_l", C.c_int32),
                ("reserved", C.c_int32)]


_P = C.c_void_p
_I64 = C.c_int64
# name -> (restype, argtypes); every symbol declared in include/vadb200.h
SIGNATURES = {
    "vadb200_last_error": (C.c_char_p, []),
    "vadb200_version": (C.c_int, []),
    "vadb200_default_config": (None, [C.POINTER(Config)]),
    "vadb200_frames_for_length": (_I64, [_I64]),
    "vadb200_outputs_for_length": (_I64, [_I64]),
    "vadb200_create": (C.c_int, [C.POINTER(Config), C.c_int, C.POINTER(_P)]),
    "vadb200_destroy": (C.c_int, [_P]),
    "vadb200_get_filterbank": (C.c_int, [_P, _P]),
    "vadb200_set_ffn_weights": (C.c_int, [_P] + [_P] * 8),
    "vadb200_set_ffn_impl": (C.c_int, [_P, C.c_int]),
    "vadb200_get_ffn_impl": (C.c_int, [_P]),
    "vadb200_set_frontend": (C.c_int, [_P, C.c_float, _P]),
    "vadb200_get_frontend": (C.c_int, [_P, _P, _P, _P]),
    "vadb200_set_decision_threshold": (C.c_int, [_P, C.c_float]),
    "vadb200_get_decision_threshold": (C.c_float, [_P]),
    "vadb200_set_tree": (C.c_int, [_P, _I64, _P, _P, _P, _P, _P, _P, C.c_int]),
    "vadb200_clear_tree": (C.c_int, [_P]),
    "vadb200_get_classifier": (C.c_int, [_P]),
    "vadb200_tree_node_count": (_I64, [_P]),
    "vadb200_tree_depth": (C.c_int, [_P]),
    "vadb200_tree_predict": (C.c_int, [_P, _P, _I64, _P, _P, _P]),
    "vadb200_plan_create": (C.c_int, [_P, _P, _P, _I64, C.c_int, C.POINTER(_P)]),
    "vadb200_plan_destroy": (C.c_int, [_P]),
    "vadb200_plan_total_rows": (_I64, [_P]),
    "vadb200_plan_row_offsets": (C.c_int, [_P, _P]),
    "vadb200_plan_segment_frames": (_I64, [_P]),
    "vadb200_plan_segment_count": (_I64, [_P]),
    "vadb200_set_plan_segment_frames": (C.c_int, [_P, C.c_int]),
    "vadb200_mfcc_host": (C.c_int, [_P, _P, _I64, _P]),
    "vadb200_plan_max_speech_segments": (_I64, [_P]),
    "vadb200_plan_speech_workspace_bytes": (_I64, [_P]),
    "vadb200_plan_speech_segments": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, _I64, _P]),
    "vadb200_plan_gather_speech": (C.c_int, [_P, _P, _I64, _P, _P, _P, _P, _I64, _P]),
    "vadb200_scale_rows": (C.c_int, [_P, _P, _I64, _P, _P]),
    "vadb200_ingest_pcm": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, C.c_int, _I64, _P, _P]),
    "vadb200_decode_pcm": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P, _P, C.c_int, _I64, _P, _P]),
    "vadb200_resampled_length": (_I64, [_I64, C.c_int]),
    "vadb200_resample_taps": (_I64, [C.c_int, _P]),
    "vadb200_resampler_create": (C.c_int, [_P, C.c_int, C.POINTER(_P)]),
    "vadb200_resampler_destroy": (C.c_int, [_P]),
    "vadb200_resample_workspace_bytes": (_I64, [_P, _I64]),
    "vadb200_resample_packed": (C.c_int, [_P, C.c_int, _P, _P, _P, _I64, _P, _I64, _P, _P, _I64, _P]),
    "vadb200_mfcc_packed": (C.c_int, [_P, _P, _I64, _P, _P]),
    "vadb200_vad_packed": (C.c_int, [_P, _P, _I64, _P, _P, _P, C.c_int, _P]),
    "vadb200_vad_host": (C.c_int, [_P, _P, _I64, _P, _P, C.c_int]),
    "vadb200_set_host_chunk_samples": (C.c_int, [_P, _I64]),
    "vadb200_spec_frames": (C.c_int, [_P, _P, _I64, C.c_int, _P, _P]),
    "vadb200_mfcc_frames": (C.c_int, [_P, _P, _I64, C.c_int, _P, _P]),
    "vadb200_mfcc_from_spec": (C.c_int, [_P, _P, _I64, _P, _P]),
    "vadb200_vad_windows": (C.c_int, [_P, _P, _I64, C.c_int, _P, _P, _P, _P]),
    "vadb200_ffn_predict": (C.c_int, [_P, _P, _I64, _P, _P, _P]),
    "vadb200_get_deltas": (C.c_int, [_P, _P, _P, _I64, _P, _P]),
    "vadb200_lifter": (C.c_int, [_P, _P, _I64, C.c_int, C.c_int, _P, _P]),
    "vadb200_stream_bank_create": (C.c_int, [_P, C.c_int, C.POINTER(_P)]),
    "vadb200_stream_bank_destroy": (C.c_int, [_P]),
    "vadb200_stream_bank_reset": (C.c_int, [_P, _P]),
    "vadb200_stream_feed": (C.c_int, [_P, _P, _P, _P, _P]),
    "vadb200_stream_bank_set_speech": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "vadb200_stream_bank_speech_delay": (C.c_int, [_P]),
    "vadb200_stream_feed_speech": (C.c_int, [_P, _P, _P, _P, _P, _P, _P]),
    "vadb200_stream_bank_end_streams": (C.c_int, [_P, _P, _P, _P, _P]),
    "vadb200_stream_bank_create_ragged": (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(_P)]),
    "vadb200_stream_bank_max_rows_per_feed": (C.c_int, [_P]),
    "vadb200_stream_feed_ragged": (C.c_int, [_P] + [_P] * 7 + [_P]),
    "vadb200_stream_bank_create_ragged_rate": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.POINTER(_P)]),
    "vadb200_stream_bank_sample_rate": (C.c_int, [_P]),
    "vadb200_trainer_create": (C.c_int, [_P, _I64, C.c_float, C.c_float, C.c_float, C.POINTER(_P)]),
    "vadb200_trainer_destroy": (C.c_int, [_P]),
    "vadb200_trainer_set_weights": (C.c_int, [_P] + [_P] * 8 + [C.c_int]),
    "vadb200_trainer_get_weights": (C.c_int, [_P] + [_P] * 8),
    "vadb200_train_on_batch": (C.c_int, [_P, _P, _P, _I64, _P, _P]),
    "vadb200_default_tree_fit_params": (None, [_P]),
    "vadb200_tree_fitter_create": (C.c_int, [_P, _I64, C.POINTER(_P)]),
    "vadb200_tree_fitter_destroy": (C.c_int, [_P]),
    "vadb200_tree_fit": (C.c_int, [_P, _P, _P, _I64, _P, _P]),
    "vadb200_tree_fit_node_count": (_I64, [_P]),
    "vadb200_tree_fit_result": (C.c_int, [_P] * 11),
    "vadb200_synth_pcm": (C.c_int, [_P, _P, _I64, _I64, _I64, C.c_uint32, _I64, _P]),
    "vadb200_fp32_peak": (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(C.c_double)]),
    "vadb200_launch_count": (_I64, []),
}

_lib = None


def load():
    """Load vad_b200/libvadb200.so (built in-tree by ``vad_b200.build``).  Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            "vad_b200: %s is missing -- build it with `python -m vad_b200.build` "
            "(nvcc, sm_100a).  There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise VadB200Error(rc, load().vadb200_last_error().decode("utf-8", "replace"))
