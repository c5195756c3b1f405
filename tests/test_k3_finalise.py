"""The utterance-mode segment scan records its finalisations and a kernel of their own (one CTA per record) runs them;
fa_segfix_kernel numbers the stores.  These cases drive every path of that finaliser -- many records, a record too large
for its shared-memory tables (finalize_segment in HBM), a dropped segment in front of stored ones, no record at all, every
output level that reads rows, and a batch in which one utterance is redone by the general kernel -- and hold each result to
the CPU oracle bit for bit."""
import sys

import numpy as np
import pytest
from conftest import GOLDEN
if GOLDEN not in sys.path:
    sys.path.insert(0, GOLDEN)

import framegen
from oracle import oracle
from webspeechanalyzer_b200 import Engine, FaConfig

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def utterance_mode(monkeypatch):
    # long test utterances would otherwise take the control-scan split (mode 1); the fast scan is the default impl
    monkeypatch.setenv("FA_K3_MODE", "0")
    monkeypatch.delenv("FA_K3_IMPL", raising=False)
    monkeypatch.delenv("FA_K3_FINALIZE_HBM", raising=False)


def run_and_compare(cfg, frames):
    """Analyse the frame blocks as one batch and compare every utterance with the oracle; returns the oracle results and
    the number of utterances the general kernel redid."""
    ans = []
    with Engine(cfg) as eng:
        for i, fr in enumerate(frames):
            eng.submit_frames(i, fr)
        eng.run()
        eng.sync()
        assert eng.counts()["overflow"] == 0
        for i, fr in enumerate(frames):
            an = oracle.analyze_frames(cfg, fr)
            r = eng.result(i)
            assert r.seg_ci == an.seg_ci, i
            # a dropped segment (stored = -1) has no store: the oracle leaves its ymax / vmin / cs_ratio at 0, the kernels
            # keep the scalars of the attempt
            kept = an.segments["stored"] >= 0
            assert np.array_equal(r.segments[kept], an.segments[kept]), i
            for name in ("start", "len", "stored", "n_syllables", "first_syllable", "row_offset"):
                assert np.array_equal(r.segments[name], an.segments[name]), (i, name)
            assert np.array_equal(r.formants, an.formants) and np.array_equal(r.energy, an.energy), i
            assert np.array_equal(r.syllables, an.syllables), i
            assert r.features.shape == an.features.shape, i
            assert np.array_equal(r.features.view(np.uint64), an.features.view(np.uint64)), i
            ans.append(an)
        redos = eng.k3_redos
    return ans, redos


def steady_comb_frames(seed, B, F):
    """F voiced frames of 13 steady peaks (one dominant) and a pause: one segment of F rows whose ~13 F points do not fit
    the finaliser's shared-memory tables once F is a few hundred."""
    rng = np.random.default_rng(seed)
    bins = np.arange(B)
    out = np.zeros((F, B))
    centres = np.arange(10, 0.68 * B, 6.0)
    for t in range(F):
        e = rng.uniform(0, 2, size=B)
        for k, c in enumerate(centres + rng.normal(0, 0.2, size=len(centres))):
            e += (4e5 if k == 3 else 2e4) * rng.uniform(0.8, 1.0) * np.exp(-0.5 * ((bins - c) / 1.0) ** 2)
        out[t] = e
    out = np.concatenate([out, rng.uniform(0, 1, size=(20, B))])
    return np.rint(out).astype(np.uint32)


def test_many_short_segments():
    cfg = FaConfig.default(output_level=13)
    frames = [framegen.voiced_random_frames(seed, cfg.bands, 3000) for seed in (11, 12)]
    ans, _ = run_and_compare(cfg, frames)
    assert min(len(an.seg_ci) for an in ans) >= 15


@pytest.mark.parametrize("hbm", [False, True])
def test_segment_too_large_for_shared_memory(hbm, monkeypatch):
    """A 320-frame segment of 13 peaks per frame (~4000 points, more than the staged tables hold) beside utterances whose
    records fit; with FA_K3_FINALIZE_HBM every record takes the HBM path."""
    if hbm:
        monkeypatch.setenv("FA_K3_FINALIZE_HBM", "1")
    cfg = FaConfig.default(output_level=13)
    frames = [steady_comb_frames(0, cfg.bands, 320), framegen.voiced_random_frames(5, cfg.bands, 400),
              steady_comb_frames(1, cfg.bands, 120)]
    ans, _ = run_and_compare(cfg, frames)
    assert int(ans[0].segments["len"].max()) == 320 and ans[0].max_peaks >= 13


def test_dropped_segment_then_stored_ones():
    cfg = FaConfig.default(output_level=13, min_seg_length_ms=25.0)
    fr = np.concatenate([framegen.dropped_segment_frames(cfg.bands), framegen.voiced_random_frames(3, cfg.bands, 600)])
    (an,), _ = run_and_compare(cfg, [fr])
    stored = an.segments["stored"]
    assert stored[0] < 0 and (stored[1:] >= 0).sum() >= 2


def test_zero_segments():
    cfg = FaConfig.default(output_level=13)
    frames = [np.zeros((120, cfg.bands), np.uint32), framegen.voiced_random_frames(8, cfg.bands, 200),
              np.zeros((1, cfg.bands), np.uint32)]
    ans, _ = run_and_compare(cfg, frames)
    assert len(ans[0].seg_ci) == 0 and len(ans[2].seg_ci) == 0 and len(ans[1].seg_ci) > 0


@pytest.mark.parametrize("level", [5, 10, 11, 12, 13])
def test_levels(level):
    cfg = FaConfig.default(output_level=level)
    frames = [framegen.voiced_random_frames(100 + u, cfg.bands, 500) for u in range(6)]
    ans, _ = run_and_compare(cfg, frames)
    assert sum(len(an.seg_ci) for an in ans) > 12


def test_batch_with_a_general_kernel_redo():
    """Comb frames with ~49 peaks each pass the fast scan's 32-peak / 64-track limits: that utterance is redone by the general
    kernel with dense rows, while its neighbours keep their rows at their epochs' first frames."""
    cfg = FaConfig.default(output_level=13, spec_type=3, n_fft_bins=256)
    frames = [framegen.voiced_random_frames(21, cfg.bands, 800), framegen.dense_peak_frames(1, cfg.bands, 300, 5.0),
              framegen.voiced_random_frames(22, cfg.bands, 800)]
    _, redos = run_and_compare(cfg, frames)
    assert redos >= 1
