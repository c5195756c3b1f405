"""Fixture for tests/test_predict.py::test_shipped_models_against_float64: the reference's shipped classifiers
(dist/nnmodel/<db>/cats_emotion: model.json + model.weights.bin + model_meta.json) scored on REAL 53-dim rows (the demo WAV
through the oracle, the app's settings: Syllable Features at 15 ms steps, and Segment Features at 25 ms) by an independent
float64 forward pass (numpy) -- ml5's min-max normalisation, Dense + relu stack, softmax.

The six shipped model directories hold three distinct weight files (4, 5, 6 and 7 are byte-identical: the fixture records
the SHA-256 of each): all three are stored, float32 bit for bit, because the GPU box has no /root/reference to read them from.
Run in the build container: python tests/golden/make_mlp_golden.py"""
import hashlib
import json
import os
import sys

import numpy as np

import npzparts

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = "/root/reference"


def forward_f64(m, rows):
    x = (np.asarray(rows, np.float64) - m["in_min"]) / (m["in_max"] - m["in_min"])
    for k, b, a in zip(m["kernels"], m["biases"], m["activations"]):
        x = x @ k.astype(np.float64) + b.astype(np.float64)
        if a == 1:
            x = np.maximum(x, 0.0)
        elif a == 2:
            x = 1.0 / (1.0 + np.exp(-x))
        elif a == 3:
            e = np.exp(x - x.max(axis=1, keepdims=True))
            x = e / e.sum(axis=1, keepdims=True)
    return x


def main():
    from oracle import oracle
    from webspeechanalyzer_b200 import FaConfig, predict, wav
    pcm, sr = wav.decode_wav(open(os.path.join(REF, "samples", "263771femaleprotagonist.wav"), "rb").read())
    rows = []
    for kw in (dict(output_level=13, window_step_ms=15.0), dict(output_level=5), dict(output_level=13)):
        _, an = oracle.analyze_pcm(FaConfig.default(**kw), pcm, sr)
        rows.append(an.features)
    rows = np.concatenate(rows)
    out = {"rows": rows}
    info = {"rows": int(rows.shape[0]), "models": {}}
    shas = {}
    for db in (1, 2, 4, 5, 6, 7):
        d = os.path.join(REF, "dist", "nnmodel", str(db), "cats_emotion")
        shas[db] = hashlib.sha256(open(os.path.join(d, "model.weights.bin"), "rb").read()).hexdigest()
    for db in (1, 2, 4):
        d = os.path.join(REF, "dist", "nnmodel", str(db), "cats_emotion")
        m = predict.load_tfjs_model(d)
        exp = forward_f64(m, rows)
        for i, (k, b) in enumerate(zip(m["kernels"], m["biases"])):
            out[f"m{db}_k{i}"], out[f"m{db}_b{i}"] = k, b
        out[f"m{db}_min"], out[f"m{db}_max"], out[f"m{db}_expected"] = m["in_min"], m["in_max"], exp
        info["models"][str(db)] = {"dims": [int(x) for x in m["dims"]], "activations": [int(a) for a in m["activations"]],
                                   "labels": m["labels"], "weights_sha256": shas[db],
                                   "same_weights_as": [k for k, v in shas.items() if v == shas[db]],
                                   "argmax_histogram": np.bincount(exp.argmax(axis=1), minlength=m["dims"][-1]).tolist()}
    npzparts.save(os.path.join(HERE, "mlp_shipped"), out)
    json.dump(info, open(os.path.join(HERE, "mlp_shipped.json"), "w"), indent=1)
    print(json.dumps(info, indent=1))


if __name__ == "__main__":
    main()
