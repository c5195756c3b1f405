"""The C-ABI library loads and exports every symbol include/fa_b200.h declares; host-only helpers work; and
without a GPU the product refuses to compute (no CPU fallback).  No compute calls here."""
import ctypes as C
import os
import re

import numpy as np

from oracle import oracle
from webspeechanalyzer_b200 import FaConfig, _capi
from webspeechanalyzer_b200._ctypes_defs import FaCounts, FaSegment, FaSyllable

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "fa_b200.h")).read()
    return re.findall(r"^FA_API\s+[\w\s\*]+?\b(fa_[a-z0-9_]+)\(", txt, flags=re.M)


def test_library_exports_every_declared_symbol():
    syms = header_symbols()
    assert len(syms) >= 30 and sorted(syms) == sorted(_capi.EXPORTS)
    L = _capi.lib()
    for s in syms:
        assert hasattr(L, s), s
    assert L.fa_abi_version() == 1


def test_synth_library_is_separate_from_the_product():
    """The workload generator lives in its own host library: a process that only generates a workload (bench.py's CPU arm)
    does not map libfa_b200.so."""
    txt = open(os.path.join(ROOT, "include", "fa_synth.h")).read()
    syms = re.findall(r"^FA_SYNTH_API\s+[\w\s\*]+?\b(fa_[a-z0-9_]+)\(", txt, flags=re.M)
    assert sorted(syms) == sorted(_capi.SYNTH_EXPORTS)
    S = _capi.synth_lib()
    for s in syms:
        assert hasattr(S, s), s
    assert not any(hasattr(_capi.lib(), s) for s in syms)
    from webspeechanalyzer_b200 import synth_speech, synth_speech_i16_batch
    a = synth_speech_i16_batch(np.zeros(3 * 8000, np.int16), 3, 8000, 16000, 5, 10, 2, threads=2).reshape(3, 8000)
    for i in range(3):
        ref = np.clip(np.rint(synth_speech(8000, 16000, 5, 10 + 2 * i).astype(np.float64) * 32768.0), -32768, 32767)
        assert np.array_equal(a[i], ref.astype(np.int16))


def test_struct_layouts_match_the_header():
    assert C.sizeof(FaSegment) == 48 and C.sizeof(FaSyllable) == 16 and C.sizeof(FaCounts) == 48
    assert C.sizeof(FaConfig) == 6 * 4 + 10 * 8 + 4 * 4 + 4 * 8
    d = FaConfig()
    _capi.lib().fa_config_default(C.byref(d))
    assert bytes(d) == bytes(FaConfig.default())   # formantanalyzer defaults @B2972 + AnalyserNode defaults


def test_host_helpers_agree_with_oracle():
    L = _capi.lib()
    for sr in (8000, 16000, 22050, 44100, 48000):
        for step in (10.0, 15.0, 25.0, 40.0):
            cfg = FaConfig.default(window_step_ms=step)
            assert L.fa_hop_samples(C.byref(cfg), sr) == oracle.hop(cfg, sr)
            assert L.fa_frames_for(C.byref(cfg), sr, 123457) == oracle.num_frames(cfg, sr, 123457)
    assert L.fa_spec_bands(C.byref(FaConfig.default())) == 128
    assert L.fa_spec_bands(C.byref(FaConfig.default(spec_type=3))) == 256


def test_synth_is_deterministic_and_bounded():
    from webspeechanalyzer_b200 import synth_speech
    a, b = synth_speech(16000, 16000, 1, 2), synth_speech(16000, 16000, 1, 2)
    assert np.array_equal(a, b) and not np.array_equal(a, synth_speech(16000, 16000, 1, 3))
    assert 0.25 < np.abs(a).max() < 0.35


NO_DEVICE_CHECK = """
import ctypes as C
from webspeechanalyzer_b200 import Engine, FaConfig, _capi
L = _capi.lib()
h = C.c_void_p()
cfg = FaConfig.default()
assert L.fa_create(C.byref(cfg), 0, C.byref(h)) == _capi.FA_ERR_NO_DEVICE and not h.value
try:
    Engine(cfg)
    raise AssertionError("Engine() without a device")
except _capi.FaError as e:
    assert e.status == _capi.FA_ERR_NO_DEVICE
"""


def test_no_cpu_fallback():
    # in a child process that sees no CUDA device, so that GPU machines check it too
    import subprocess
    import sys
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    subprocess.run([sys.executable, "-c", NO_DEVICE_CHECK], cwd=ROOT, env=env, check=True)


def test_product_never_touches_the_oracle():
    """The product package must not import, load or link anything under oracle/."""
    pkg = os.path.join(ROOT, "webspeechanalyzer_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h", ".c", ".js")):
                txt = open(os.path.join(dp, f), errors="ignore").read()
                assert "oracle" not in txt.replace("the CPU oracle", "").replace("oracle/fa_oracle.c", "").replace("oracle's", "").replace("the oracle", ""), (dp, f)
