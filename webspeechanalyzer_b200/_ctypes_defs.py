"""ctypes mirrors of the plain-C structs in include/fa_b200.h (no library is loaded here)."""
from __future__ import annotations

import ctypes as C

N_FEATURES = 53  # /root/reference/src/localstore.js:7
SPECTRUM_F32, SPECTRUM_U8, SPECTRUM_F16 = 0, 1, 2   # fa_config.spectrum_format
N_CURVE_FEATURES = 23  # /root/reference/src/localstore.js:7 (level 12): make_coeffs @B34527
N_UTT_FEATURES = 264  # get_utterance_features, /root/reference/dist/main.js:2@B107983 (level 11)


class FaConfig(C.Structure):
    _fields_ = [
        ("spec_type", C.c_int32), ("output_level", C.c_int32), ("plot_len", C.c_int32), ("n_fft_bins", C.c_int32),
        ("n_mel_bins", C.c_int32), ("auto_noise_gate", C.c_int32),
        ("f_min", C.c_double), ("f_max", C.c_double), ("window_width_ms", C.c_double), ("window_step_ms", C.c_double),
        ("pause_length_ms", C.c_double), ("min_seg_length_ms", C.c_double), ("voiced_max_db", C.c_double),
        ("voiced_min_db", C.c_double), ("pre_norm_gain", C.c_double), ("high_f_emph", C.c_double),
        ("fft_size", C.c_int32), ("clamp_db", C.c_int32), ("want_spectrum", C.c_int32), ("spectrum_format", C.c_int32),
        ("smoothing", C.c_double), ("min_db", C.c_double), ("max_db", C.c_double), ("mag_scale", C.c_double),
    ]

    @classmethod
    def default(cls, **over) -> "FaConfig":
        """formantanalyzer defaults (/root/reference/dist/main.js:2@B2972) + AnalyserNode defaults (W3C)."""
        c = cls(spec_type=1, output_level=4, plot_len=200, n_fft_bins=256, n_mel_bins=128, auto_noise_gate=1,
                f_min=50.0, f_max=4000.0, window_width_ms=25.0, window_step_ms=25.0, pause_length_ms=200.0,
                min_seg_length_ms=50.0, voiced_max_db=100.0, voiced_min_db=10.0, pre_norm_gain=1000.0, high_f_emph=0.0,
                fft_size=2048, clamp_db=1, want_spectrum=0, spectrum_format=0, smoothing=0.8, min_db=-100.0, max_db=-30.0,
                mag_scale=0.0)
        for k, v in over.items():
            if not hasattr(c, k):
                raise AttributeError(k)
            setattr(c, k, v)
        return c

    def copy(self) -> "FaConfig":
        c = FaConfig()
        C.memmove(C.byref(c), C.byref(self), C.sizeof(FaConfig))
        return c

    @property
    def bands(self) -> int:
        return self.n_mel_bins if self.spec_type == 1 else self.n_fft_bins


class FaSegment(C.Structure):
    _fields_ = [("start", C.c_int32), ("len", C.c_int32), ("stored", C.c_int32), ("n_syllables", C.c_int32),
                ("first_syllable", C.c_int32), ("row_offset", C.c_int32), ("ymax", C.c_double), ("vmin", C.c_double),
                ("cs_ratio", C.c_double)]


class FaSyllable(C.Structure):
    _fields_ = [("stored_seg", C.c_int32), ("start", C.c_int32), ("len", C.c_int32), ("reserved", C.c_int32)]


class FaCounts(C.Structure):
    _fields_ = [("samples", C.c_int64), ("sample_rate", C.c_int32), ("hop", C.c_int32), ("frames", C.c_int32),
                ("bands", C.c_int32), ("segments", C.c_int32), ("stored_segments", C.c_int32),
                ("formant_rows", C.c_int32), ("syllables", C.c_int32), ("feature_rows", C.c_int32),
                ("overflow", C.c_int32)]


class FaTrainOpts(C.Structure):
    _fields_ = [("learning_rate", C.c_double), ("optimizer", C.c_int32), ("epochs", C.c_int32), ("batch_size", C.c_int32)]
