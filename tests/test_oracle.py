"""The CPU oracle: against the committed golden vectors, against the literal transliteration of the reference's
modules (oracle/literal/refmodules.py) and against the invariants the reference pins (SURVEY.md section 4)."""
import json
import os
import sys

import numpy as np
import pytest
from conftest import GOLDEN, sha
from hypothesis import given, settings, strategies as st

sys.path.insert(0, GOLDEN)
import npzparts  # noqa: E402
from framegen import adversarial_frames, voiced_random_frames  # noqa: E402

from oracle import oracle  # noqa: E402
from oracle.literal.refmodules import Segmentor, toFixed3
from webspeechanalyzer_b200 import FaConfig, synth_speech

SURVEY_APPENDIX_D = [(87, 68), (254, 90), (431, 120), (640, 95), (837, 32), (903, 85), (1090, 88), (1279, 71),
                     (1451, 94), (1627, 83), (1799, 72), (1958, 103)]


def literal(cfg: FaConfig, frames: np.ndarray) -> Segmentor:
    S = Segmentor(cfg.output_level, cfg.bands, cfg.plot_len, cfg.window_step_ms, cfg.pause_length_ms,
                  cfg.min_seg_length_ms, bool(cfg.auto_noise_gate), cfg.voiced_max_db, cfg.voiced_min_db, None, True, [])
    for f in frames:
        S.spectrum_push(f)
    S.segment_truncate()
    return S


def assert_same(S: Segmentor, an, level):
    assert [tuple(x) for x in S.u] == an.seg_ci
    if level >= 4:
        Fl = np.concatenate([np.stack(c) for c in S.c if len(c)]) if any(len(c) for c in S.c) else np.zeros((0, 9), np.float32)
        assert np.array_equal(Fl, an.formants)
    if level in (10, 13):
        syl = [(k, s[0], s[1]) for k, h in enumerate(S.h) for s in h[0]]
        assert syl == [(int(s["stored_seg"]), int(s["start"]), int(s["len"])) for s in an.syllables]
    if level == 13:
        rows = np.array([r for p in S.p for r in p]).reshape(-1, 53)
        assert np.array_equal(rows, an.features, equal_nan=True)
    if level == 5:
        assert np.array_equal(np.array(S.d).reshape(-1, 53), an.features, equal_nan=True)
    assert [e[0] for e in S.events] == an.callbacks.tolist()


# ------------------------------------------------------------------ golden vectors
def test_sample_wav_full_file_pins(sample_full):
    c = sample_full["configs"]["app_l13_step15"]
    assert [tuple(x) for x in c["seg_ci"]] == SURVEY_APPENDIX_D  # SURVEY.md Appendix D, tau=0.8, scale N, level 13
    assert c["frames"] == 2110 and c["max_band"] == 60671
    assert c["last_row_head"][0] == 101 and abs(c["last_row_head"][3] - 4.21) < 5e-3 and c["last_row_head"][4] == 13
    assert abs(c["last_row_head"][2] - 7.621) < 1e-3
    assert len(sample_full["configs"]["default_l5_step25"]["seg_ci"]) == 12


@pytest.mark.parametrize("name,kw", [("app_l13_step15", dict(output_level=13, window_step_ms=15.0)),
                                     ("default_l5_step25", dict(output_level=5, window_step_ms=25.0))])
def test_oracle_reproduces_sample_excerpt(sample_excerpt, name, kw):
    g = sample_excerpt
    pcm = g["pcm_i16"].astype(np.float32) / 32768.0
    cfg = FaConfig.default(**kw)
    fe, an = oracle.analyze_pcm(cfg, pcm, int(g["sample_rate"]))
    assert np.array_equal(fe["frames"], g[f"{name}/frames"])
    assert np.array_equal(np.array(an.seg_ci, np.int32).reshape(-1, 2), g[f"{name}/seg_ci"])
    assert np.array_equal(an.formants, g[f"{name}/formants"])
    assert np.array_equal(an.energy, g[f"{name}/energy"])
    assert np.array_equal(an.features, g[f"{name}/features"], equal_nan=True)
    # the literal transliteration agrees on the same frames
    assert_same(literal(cfg, fe["frames"]), an, cfg.output_level)


def test_synth_golden(synth_golden):
    for c in synth_golden["cases"]:
        p = synth_speech(c["seconds"] * c["sample_rate"], c["sample_rate"], c["seed"], c["utt"])
        assert sha(p) == c["pcm_sha"]
        cfg = FaConfig.default(**c["kwargs"])
        fe, an = oracle.analyze_pcm(cfg, p, c["sample_rate"])
        assert sha(fe["frames"]) == c["frames_sha"]
        assert an.seg_ci == [tuple(x) for x in c["seg_ci"]]
        assert sha(an.features) == c["features_sha"] and sha(an.formants) == c["formants_sha"]


# ------------------------------------------------------------------ what the reference pins
def test_row_width_and_identities():
    # /root/reference/src/localstore.js:7 -> level 5 and 13 rows have 53 entries; f[1] == sqrt(f[0])
    for lvl in (5, 13):
        cfg = FaConfig.default(output_level=lvl)
        _, an = oracle.analyze_pcm(cfg, synth_speech(5 * 16000, 16000, 3, lvl), 16000)
        assert an.features.shape[1] == 53 and an.features.shape[0] > 0
        assert np.array_equal(an.features[:, 1], np.sqrt(an.features[:, 0]))
        for k in (20, 36, 52):
            assert ((an.features[:, k] >= 0) & (an.features[:, k] <= 100)).all()


def test_feature_ranges_against_model_meta(sample_full):
    # the input ranges of the app's model 1 (dist/nnmodel/1/cats_emotion/model_meta.json, stored by make_mlp_golden.py)
    # and the demo WAV's PCM (make_golden.py)
    meta = npzparts.load(os.path.join(GOLDEN, "mlp_shipped"))
    wav = npzparts.load(os.path.join(GOLDEN, "sample_full_pcm"))
    pcm = wav["pcm_i16"].astype(np.float32) / 32768.0
    _, an = oracle.analyze_pcm(FaConfig.default(output_level=13, window_step_ms=15.0), pcm, int(wav["sample_rate"]))
    lo, hi = meta["m1_min"], meta["m1_max"]
    # the real-data ranges of 74 249 syllables bound ours on the demo file (small slack on the open-ended ones)
    inside = (an.features >= lo - 1e-9) & (an.features <= hi * 1.25 + 1e-9)
    assert inside.mean() > 0.99, np.argwhere(~inside)


# ------------------------------------------------------------------ restatement vs literal transliteration
@pytest.mark.parametrize("level", [4, 5, 10, 13])
@pytest.mark.parametrize("sr,step", [(16000, 25.0), (48000, 25.0), (44100, 15.0)])
def test_oracle_equals_literal_on_synth(level, sr, step):
    cfg = FaConfig.default(output_level=level, window_step_ms=step)
    for u in range(2):
        fe, an = oracle.analyze_pcm(cfg, synth_speech(4 * sr, sr, 11, u), sr)
        assert_same(literal(cfg, fe["frames"]), an, level)


frames_strategy = st.integers(0, 2 ** 31).flatmap(lambda seed: st.just(seed))


@settings(max_examples=25, deadline=None)
@given(seed=st.integers(0, 2 ** 31), B=st.sampled_from([32, 128, 256]), F=st.integers(1, 120),
       auto=st.booleans(), level=st.sampled_from([4, 5, 13]))
def test_oracle_equals_literal_on_random_frames(seed, B, F, auto, level):
    """Adversarial frames: smooth random spectra with moving bumps, silences and huge / tiny amplitudes (and, every other
    example, runs of voiced frames that do open and close segments)."""
    frames = voiced_random_frames(seed, B, F) if seed % 2 else adversarial_frames(seed, B, F)
    cfg = FaConfig.default(output_level=level, auto_noise_gate=int(auto), voiced_max_db=100.0, voiced_min_db=30.0)
    cfg.n_mel_bins = B
    an = oracle.analyze_frames(cfg, frames)
    assert_same(literal(cfg, frames), an, level)


# ------------------------------------------------------------------ stage-2 decoupling (SURVEY.md A.3)
@settings(max_examples=200, deadline=None)
@given(seed=st.integers(0, 2 ** 31), B=st.sampled_from([16, 128, 256]), v=st.sampled_from([0.5, 2.0, 10.0, 100.0, 3.1622776601683795]))
def test_candidates_filtered_by_v_equal_literal_scan(seed, B, v):
    rng = np.random.default_rng(seed)
    e = np.rint(np.abs(rng.normal(0, 1, B)).cumsum() % 50 * rng.choice([0, 1, 1, 20])).astype(np.uint32)
    if seed % 3 == 0:
        e = rng.integers(0, 40, B).astype(np.uint32)
    packed, g = oracle.peak_candidates(e)
    cand = [(int(p & 0xff), int((p >> 8) & 0xff), int((p >> 16) & 0xff), int(p >> 24)) for p in packed]
    keep = [(lo, hi, pk) for lo, hi, pk, _ in cand if e[pk] > v]
    # literal scan with threshold v: run one frame through the transliteration and read its peak list back
    S = Segmentor(4, B, auto_noise_gate=False, voiced_max_dB=100, voiced_min_dB=20)
    S.v = v
    peaks = []
    orig = S.r.accumulate_fm
    S.r.accumulate_fm = lambda e_, f, *a: peaks.extend(map(tuple, f))
    S.o["c_started"] = 5  # force the voiced branch to reach accumulate_fm when the frame is voiced
    S.o["max_voiced_bin"] = 10 ** 9
    S._D_frame([int(x) for x in e])
    n, h, p = S.trace[-1][0], S.trace[-1][1], S.trace[-1][2]
    assert n == len(keep)
    assert g == float(e[1:].astype(np.float64).sum())
    nonlast = [(e[pk], i) for i, (lo, hi, pk, last) in enumerate(c for c in cand if e[c[2]] > v) if not last]
    hh = max([2 * v] + [float(a) for a, _ in nonlast])
    assert h == hh
    if peaks:
        assert peaks == keep
    S.r.accumulate_fm = orig


# ------------------------------------------------------------------ front end
def test_frame_count_and_hop_rule():
    cfg = FaConfig.default()
    assert oracle.hop(cfg, 44100) == 1103      # Math.round(1102.5) -> 1103
    assert oracle.hop(cfg, 16000) == 400 and oracle.hop(cfg, 48000) == 1200
    cfg.window_step_ms = 15.0
    assert oracle.hop(cfg, 44100) == 662
    assert oracle.num_frames(cfg, 44100, 1396908) == 2110
    assert oracle.frontend(cfg, np.zeros(100, np.float32), 44100)["frames"].shape == (0, 128)


def test_float32_front_end_close_to_float64_truth():
    sr = 16000
    p = synth_speech(2 * sr, sr, 5, 0)
    cfg = FaConfig.default(clamp_db=0)
    s32 = oracle.frontend(cfg, p, sr)["spectrum"].astype(np.float64)
    s64 = oracle.frontend_f64(cfg, p, sr)
    peak = s64.max(axis=1, keepdims=True)
    strong = s64 > peak - 60.0          # bins within 60 dB of the frame peak
    assert np.abs(s32 - s64)[strong].max() < 2e-2
    assert np.abs(s32 - s64)[s64 > peak - 30.0].max() < 2e-3


def test_power_of_two_scaling_is_exact():
    """All float32 ops of the canonical DAG commute with scaling by 2^k (no under/overflow here)."""
    sr = 16000
    p = synth_speech(sr, sr, 6, 0)
    cfg = FaConfig.default()
    a = oracle.frontend(cfg, p, sr, smooth=True)["smooth"]
    b = oracle.frontend(cfg, (p * np.float32(0.25)), sr, smooth=True)["smooth"]
    assert np.array_equal(a * np.float32(0.25), b)


def test_smoothing_recursion():
    sr = 16000
    p = synth_speech(sr, sr, 8, 0)
    c0 = FaConfig.default(smoothing=0.0)
    c8 = FaConfig.default(smoothing=0.8)
    m = oracle.frontend(c0, p, sr, smooth=True)["smooth"]
    s = oracle.frontend(c8, p, sr, smooth=True)["smooth"]
    tau, omt = np.float32(0.8), np.float32(1.0 - 0.8)
    x = np.zeros(m.shape[1], np.float64)
    for t in range(m.shape[0]):
        x = tau.astype(np.float64) * x + (omt * m[t]).astype(np.float64)   # fma in double then one rounding
        x = x.astype(np.float32).astype(np.float64)
        assert np.array_equal(x.astype(np.float32), s[t])


def test_to_fixed3():
    assert toFixed3(0.0625) == "0.063"      # JS picks the larger n on ties; printf would give 0.062
    assert toFixed3(1.005) == "1.005" and toFixed3(2.5) == "2.500" and toFixed3(0.0004) == "0.000"
