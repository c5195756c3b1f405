"""Regenerates the golden fixtures in this directory.  Run in the build container (needs /root/reference):

    python tests/golden/make_golden.py

* sample_excerpt.npz : the first 10 s of /root/reference/samples/263771femaleprotagonist.wav (int16 mono 44.1 kHz,
  BASELINE.json config #1 input) and what the CPU oracle produces from it (uint32 frames, seg_ci, formant rows,
  syllables, 53-dim rows) for the app's settings (/root/reference/src/index.js:21: level 13, step 15 ms) and for the
  formantanalyzer defaults at level 5 (step 25 ms).
* sample_full.json   : pins over the WHOLE file: seg_ci for both settings (the level-13 list equals the one a
  survey-time transliteration printed, SURVEY.md Appendix D), row counts, and checksums of frames / features.
* synth.json         : oracle results for seeded synthetic utterances (guards the generator and the oracle
  against drift; the -m gpu tests compare the CUDA path with these too).

The reference ships no golden vectors and cannot run here (browser JS, no JS engine), so these vectors come from
the restated oracle: they pin the oracle against regressions, not against the reference.
"""
from __future__ import annotations

import hashlib
import json
import os
import sys
import wave

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import npzparts  # noqa: E402
from oracle import oracle  # noqa: E402
from webspeechanalyzer_b200 import FaConfig  # noqa: E402
from webspeechanalyzer_b200.engine import synth_speech  # noqa: E402

WAV = "/root/reference/samples/263771femaleprotagonist.wav"
CONFIGS = {
    "app_l13_step15": dict(output_level=13, window_step_ms=15.0),
    "default_l5_step25": dict(output_level=5, window_step_ms=25.0),
}


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def run(cfg_kw, pcm, sr):
    cfg = FaConfig.default(**cfg_kw)
    fe, an = oracle.analyze_pcm(cfg, pcm, sr)
    return cfg, fe, an


def main():
    w = wave.open(WAV)
    sr, n = w.getframerate(), w.getnframes()
    i16 = np.frombuffer(w.readframes(n), np.int16)
    pcm = i16.astype(np.float32) / 32768.0
    exc = i16[: 10 * sr]
    out = {"pcm_i16": exc, "sample_rate": np.int32(sr)}
    full = {"wav": os.path.basename(WAV), "samples": int(n), "sample_rate": int(sr), "configs": {}}
    for name, kw in CONFIGS.items():
        _, fe, an = run(kw, exc.astype(np.float32) / 32768.0, sr)
        out[f"{name}/frames"] = fe["frames"]
        out[f"{name}/seg_ci"] = np.array(an.seg_ci, np.int32).reshape(-1, 2)
        out[f"{name}/formants"] = an.formants
        out[f"{name}/energy"] = an.energy
        out[f"{name}/syllables"] = np.array([(s["stored_seg"], s["start"], s["len"]) for s in an.syllables], np.int32).reshape(-1, 3)
        out[f"{name}/features"] = an.features
        _, fe, an = run(kw, pcm, sr)
        full["configs"][name] = {
            "kwargs": kw, "frames": int(fe["frames"].shape[0]), "max_band": int(fe["frames"].max()),
            "frames_sha": sha(fe["frames"]), "seg_ci": an.seg_ci, "syllables": len(an.syllables),
            "feature_rows": int(an.features.shape[0]), "features_sha": sha(an.features),
            "formants_sha": sha(an.formants), "syllable_table": [(int(y["stored_seg"]), int(y["start"]), int(y["len"])) for y in an.syllables],
            "last_row_head": [float(x) for x in an.features[-1][:6]],
        }
    np.savez_compressed(os.path.join(HERE, "sample_excerpt.npz"), **out)
    # the whole demo file (BASELINE config 1 input) as int16, so that the -m gpu tests can run C1 in full on the GPU
    # box, where /root/reference does not exist
    npzparts.save(os.path.join(HERE, "sample_full_pcm"), {"pcm_i16": i16, "sample_rate": np.int32(sr)})
    json.dump(full, open(os.path.join(HERE, "sample_full.json"), "w"), indent=1)

    synth = {"cases": []}
    for sr_, secs, seed, utt, kw in [(16000, 5, 1, 0, dict(output_level=13)), (16000, 5, 1, 3, dict(output_level=5)),
                                     (48000, 5, 7, 11, dict(output_level=13)), (44100, 4, 2, 5, dict(output_level=4, window_step_ms=15.0)),
                                     (16000, 5, 9, 2, dict(output_level=13, fft_size=1024, smoothing=0.0)),
                                     (16000, 3, 4, 1, dict(output_level=5, spec_type=3, fft_size=512))]:
        p = synth_speech(secs * sr_, sr_, seed, utt)
        cfg, fe, an = run(kw, p, sr_)
        synth["cases"].append({"sample_rate": sr_, "seconds": secs, "seed": seed, "utt": utt, "kwargs": kw,
                               "pcm_sha": sha(p), "frames_sha": sha(fe["frames"]), "seg_ci": an.seg_ci,
                               "syllables": [(int(s["stored_seg"]), int(s["start"]), int(s["len"])) for s in an.syllables],
                               "features_sha": sha(an.features), "formants_sha": sha(an.formants)})
    json.dump(synth, open(os.path.join(HERE, "synth.json"), "w"), indent=1)
    print("wrote", os.listdir(HERE))


if __name__ == "__main__":
    main()
