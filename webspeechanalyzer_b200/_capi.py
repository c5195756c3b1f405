"""ctypes binding of libfa_b200.so -- the C-ABI declared in include/fa_b200.h.

There is deliberately no fallback: if the CUDA library is missing this module raises, and if no
sm_100 device is present fa_create returns FA_ERR_NO_DEVICE (surfaced as FaError).
"""
from __future__ import annotations

import ctypes as C
import os

from ._ctypes_defs import FaConfig, FaCounts, FaSegment, FaSyllable, FaTrainOpts

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfa_b200.so")

FA_OK = 0
FA_ERR_INVALID_ARG, FA_ERR_NO_DEVICE, FA_ERR_CUDA, FA_ERR_NOT_RUN, FA_ERR_UNKNOWN_UTT = -1, -2, -3, -4, -5
FA_ERR_CAPACITY, FA_ERR_OUT_OF_MEMORY, FA_ERR_BUSY, FA_ERR_UNSUPPORTED = -6, -7, -8, -9

# every symbol include/fa_b200.h declares (tests check that the library exports all of them)
EXPORTS = [
    "fa_config_default", "fa_abi_version", "fa_status_string", "fa_create", "fa_destroy", "fa_last_error", "fa_get_config",
    "fa_set_stream", "fa_set_d2h_stream", "fa_set_pipeline", "fa_set_spectrum_sink", "fa_set_spectrum_sink_raw", "fa_reset", "fa_submit_pcm", "fa_submit_pcm_i16", "fa_submit_pcm_batch", "fa_submit_pcm_i16_batch", "fa_submit_frames", "fa_run", "fa_sync", "fa_upload",
    "fa_run_resident", "fa_download", "fa_stage_times", "fa_spectrum_split_times", "fa_launch_count", "fa_stream_fixups", "fa_num_utterances", "fa_result_counts",
    "fa_total_counts", "fa_copy_counts_table", "fa_pcie_probe", "fa_copy_spectrum", "fa_copy_spectrum_raw", "fa_copy_frames", "fa_copy_segments", "fa_copy_formants", "fa_copy_energy",
    "fa_copy_syllables", "fa_copy_features", "fa_copy_utterance_features", "fa_copy_curve_features", "fa_copy_track_points", "fa_set_truncate", "fa_mlp_create", "fa_mlp_destroy", "fa_mlp_last_error",
    "fa_mlp_classify", "fa_mlp_classify_features", "fa_copy_peak_candidates", "fa_copy_gsum", "fa_hop_samples", "fa_frames_for",
    "fa_spec_bands", "fa_host_alloc", "fa_host_free", "fa_mlp_train",
]
SYNTH_EXPORTS = ["fa_synth_speech", "fa_synth_speech_i16_batch"]   # include/fa_synth.h -> libfa_synth.so (host-only generator)


class FaError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"fa_b200 status {status}: {message}")
        self.status = status
        self.message = message


_lib = None


def lib() -> C.CDLL:
    """Load libfa_b200.so (built in-tree by webspeechanalyzer_b200/build.py).  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m webspeechanalyzer_b200.build` "
            "(or __graft_entry__.build()).  There is no CPU fallback for the hot path.")
    L = C.CDLL(LIB_PATH)
    H = C.c_void_p
    cfgp = C.POINTER(FaConfig)
    L.fa_config_default.argtypes = [cfgp]; L.fa_config_default.restype = None
    L.fa_abi_version.restype = C.c_int
    L.fa_status_string.argtypes = [C.c_int]; L.fa_status_string.restype = C.c_char_p
    L.fa_create.argtypes = [cfgp, C.c_int, C.POINTER(H)]
    L.fa_destroy.argtypes = [H]
    L.fa_last_error.argtypes = [H]; L.fa_last_error.restype = C.c_char_p
    L.fa_get_config.argtypes = [H, cfgp]
    L.fa_set_stream.argtypes = [H, C.c_void_p]
    L.fa_set_d2h_stream.argtypes = [H, C.c_void_p]
    L.fa_reset.argtypes = [H]
    L.fa_submit_pcm.argtypes = [H, C.c_int64, C.c_void_p, C.c_size_t, C.c_int]
    L.fa_submit_pcm_i16.argtypes = [H, C.c_int64, C.c_void_p, C.c_size_t, C.c_int]
    L.fa_submit_pcm_batch.argtypes = [H, C.c_int64, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    L.fa_submit_pcm_i16_batch.argtypes = [H, C.c_int64, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    L.fa_submit_frames.argtypes = [H, C.c_int64, C.c_void_p, C.c_size_t, C.c_int]
    L.fa_set_pipeline.argtypes = [H, C.c_int]
    L.fa_set_truncate.argtypes = [H, C.c_int]
    L.fa_set_spectrum_sink.argtypes = [H, C.c_void_p, C.c_size_t]
    L.fa_set_spectrum_sink_raw.argtypes = [H, C.c_void_p, C.c_size_t]
    for n in ("fa_run", "fa_sync", "fa_upload", "fa_run_resident", "fa_download", "fa_launch_count", "fa_num_utterances"):
        getattr(L, n).argtypes = [H]
    L.fa_stream_fixups.argtypes = [H, C.c_int]
    L.fa_stage_times.argtypes = [H, C.POINTER(C.c_float)]
    L.fa_spectrum_split_times.argtypes = [H, C.POINTER(C.c_float)]
    L.fa_result_counts.argtypes = [H, C.c_int64, C.POINTER(FaCounts)]
    L.fa_total_counts.argtypes = [H, C.POINTER(FaCounts)]
    L.fa_copy_counts_table.argtypes = [H, C.c_void_p, C.c_size_t]
    L.fa_pcie_probe.argtypes = [C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.POINTER(C.c_float)]
    for n in ("fa_copy_gsum", "fa_copy_spectrum", "fa_copy_spectrum_raw", "fa_copy_frames", "fa_copy_segments", "fa_copy_formants", "fa_copy_energy",
              "fa_copy_syllables", "fa_copy_features", "fa_copy_utterance_features", "fa_copy_curve_features", "fa_copy_track_points"):
        getattr(L, n).argtypes = [H, C.c_int64, C.c_void_p, C.c_size_t]
    L.fa_mlp_create.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(H)]
    L.fa_mlp_destroy.argtypes = [H]
    L.fa_mlp_last_error.argtypes = [H]; L.fa_mlp_last_error.restype = C.c_char_p
    L.fa_mlp_classify.argtypes = [H, C.c_void_p, C.c_size_t, C.c_void_p]
    L.fa_mlp_classify_features.argtypes = [H, H, C.c_int64, C.c_void_p, C.c_size_t]
    L.fa_mlp_train.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(FaTrainOpts), C.c_int,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_char_p, C.c_size_t]
    L.fa_copy_peak_candidates.argtypes = [H, C.c_int64, C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_int32)]
    L.fa_hop_samples.argtypes = [cfgp, C.c_int]
    L.fa_frames_for.argtypes = [cfgp, C.c_int, C.c_size_t]
    L.fa_spec_bands.argtypes = [cfgp]
    L.fa_host_alloc.argtypes = [C.c_size_t, C.c_int]; L.fa_host_alloc.restype = C.c_void_p
    L.fa_host_free.argtypes = [C.c_void_p]; L.fa_host_free.restype = None
    _lib = L
    return L


_synth = None
SYNTH_LIB_PATH = os.path.join(_HERE, "libfa_synth.so")


def synth_lib() -> C.CDLL:
    """The host-only workload generator (csrc/fa_synth.cpp); a separate library, so that generating a workload -- e.g. for a
    CPU baseline -- never maps the CUDA library."""
    global _synth
    if _synth is None:
        if not os.path.exists(SYNTH_LIB_PATH):
            raise ImportError(f"{SYNTH_LIB_PATH} is missing: build it with `python -m webspeechanalyzer_b200.build`")
        S = C.CDLL(SYNTH_LIB_PATH)
        S.fa_synth_speech.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_uint64, C.c_uint64]
        S.fa_synth_speech_i16_batch.argtypes = [C.c_void_p, C.c_int, C.c_size_t, C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int]
        _synth = S
    return _synth
