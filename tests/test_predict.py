"""The web app's classifier path (SURVEY 8(f) rank 3): tf.js model loading, ml5 result shapes and the sqrt(duration) vote on
CPU; the CUDA forward pass against a plain float32 loop on the GPU (tolerance 1e-5 on the class scores: tf.js's own
summation order is unspecified, so bit parity with the app is not defined for this stage)."""
import json
import os

import numpy as np
import pytest

from webspeechanalyzer_b200 import predict


def write_model(tmp, dims=(53, 256, 64, 16, 4), acts=("relu", "relu", "relu", "softmax"), seed=0):
    rng = np.random.default_rng(seed)
    layers, weights, blob = [], [], b""
    for i, (a, b) in enumerate(zip(dims[:-1], dims[1:])):
        name = f"dense_Dense{i + 5}"
        cfg = {"units": b, "activation": acts[i], "use_bias": True, "name": name}
        if i == 0:
            cfg["batch_input_shape"] = [None, a]
        layers.append({"class_name": "Dense", "config": cfg})
        k = (rng.normal(0, 1.5 / np.sqrt(a), (a, b))).astype("<f4")
        bias = rng.normal(0, 0.1, b).astype("<f4")
        weights += [{"name": name + "/kernel", "shape": [a, b], "dtype": "float32"}, {"name": name + "/bias", "shape": [b], "dtype": "float32"}]
        blob += k.tobytes() + bias.tobytes()
    doc = {"modelTopology": {"class_name": "Sequential", "config": {"name": "sequential_3", "layers": layers}},
           "weightsManifest": [{"paths": ["./model.weights.bin"], "weights": weights}]}
    labs = ["N", "A", "S", "H"][: dims[-1]]
    meta = {"inputUnits": [dims[0]], "outputUnits": dims[-1],
            "inputs": {str(i): {"dtype": "number", "min": float(-i), "max": float(10 + 3 * i)} for i in range(dims[0])},
            "outputs": {"y": {"dtype": "string", "uniqueValues": labs,
                              "legend": {l: [1 if j == i else 0 for j in range(len(labs))] for i, l in enumerate(labs)}}}}
    os.makedirs(tmp, exist_ok=True)
    json.dump(doc, open(os.path.join(tmp, "model.json"), "w"))
    json.dump(meta, open(os.path.join(tmp, "model_meta.json"), "w"))
    open(os.path.join(tmp, "model.weights.bin"), "wb").write(blob)
    return tmp


def forward_f32(m, rows):
    """Plain float32 loop in index order (the kernel's DAG, minus fused multiply-add)."""
    x = ((np.asarray(rows, np.float64) - m["in_min"]) / (m["in_max"] - m["in_min"])).astype(np.float32)
    for k, b, a in zip(m["kernels"], m["biases"], m["activations"]):
        acc = np.zeros((x.shape[0], k.shape[1]), np.float32)
        for i in range(k.shape[0]):
            acc = (acc + x[:, i: i + 1] * k[i: i + 1, :]).astype(np.float32)
        v = (acc + b).astype(np.float32)
        if a == 1:
            v = np.where(v > 0, v, np.where(np.isnan(v), v, 0)).astype(np.float32)
        elif a == 2:
            v = (1 / (1 + np.exp(-v))).astype(np.float32)
        elif a == 3:
            e = np.exp(v - v.max(axis=1, keepdims=True)).astype(np.float32)
            v = (e / e.sum(axis=1, keepdims=True)).astype(np.float32)
        x = v
    return x


def test_tfjs_loader_reads_the_layers_format(tmp_path):
    m = predict.load_tfjs_model(write_model(str(tmp_path)))
    assert m["dims"] == [53, 256, 64, 16, 4] and m["activations"] == [1, 1, 1, 3] and m["labels"] == ["N", "A", "S", "H"]
    assert m["kernels"][0].shape == (53, 256) and m["biases"][3].shape == (4,) and m["in_max"][2] == 16.0
    ref = "/root/reference/dist/nnmodel/1/cats_emotion"
    if os.path.exists(ref):       # the web app's own model files load (read in place, nothing copied)
        r = predict.load_tfjs_model(ref)
        assert r["dims"] == [53, 256, 64, 16, 4] and r["labels"] == ["N", "A", "S", "H"] and r["in_min"][0] == 2
        p = forward_f32(r, np.stack([r["in_min"], r["in_max"], (r["in_min"] + r["in_max"]) / 2]))
        assert p.shape == (3, 4) and np.allclose(p.sum(axis=1), 1, atol=1e-5)


def test_segment_vote_follows_prediction_js():
    # two syllables: every label of every syllable adds confidence * sqrt(duration)   (src/prediction.js:106-116)
    res = [[{"label": "H", "confidence": 0.6}, {"label": "N", "confidence": 0.4}],
           [{"label": "N", "confidence": 0.7}, {"label": "H", "confidence": 0.3}]]
    v = predict.SegmentVoter([1])
    top, conf = v.segment({1: res}, [["0.100", "0.250"], ["0.400", "1.000"]])
    n = 0.4 * 0.5 + 0.7 * 1.0
    h = 0.6 * 0.5 + 0.3 * 1.0
    assert top == "N" and abs(conf - n / 1.25) < 1e-12 and abs(v.conf_all[1]["H"] - h) < 1e-12
    # one syllable: only the top class is counted (the app indexes the flat class list, src/prediction.js:96-103)
    top, conf = v.segment({1: [res[0]]}, [["2.000", "0.640"]])
    assert top == "H" and abs(conf - 0.6 * 0.8 / 0.64) < 1e-12
    assert abs(v.conf_all[1]["H"] - (h + 0.48)) < 1e-12 and v.min_entropy_db == 1 and abs(v.sum_weights - 1.89) < 1e-12
    assert v.segment({1: []}, []) is None


@pytest.mark.gpu
def test_mlp_kernel_matches_float32_loop(tmp_path):
    m = predict.load_tfjs_model(write_model(str(tmp_path)))
    clf = predict.Classifier(m)
    rng = np.random.default_rng(1)
    rows = rng.uniform(-5, 60, (1003, 53))
    rows[7, 3] = np.nan                                   # NaN features propagate like in tf.js
    p = clf.probabilities(rows)
    ref = forward_f32(m, rows)
    ok = ~np.isnan(ref).any(axis=1)
    assert not ok[7] and np.isnan(p[7]).all()
    assert np.abs(p[ok] - ref[ok]).max() < 1e-5 and np.allclose(p[ok].sum(axis=1), 1, atol=1e-5)
    r = clf.classify_multiple(rows[:3])
    assert [x["label"] for x in r[0]] == [clf.labels[i] for i in np.argsort(-p[0], kind="stable")]
    assert clf.probabilities(np.zeros((0, 53))).shape == (0, 4)
    # other shapes / activations
    m2 = predict.load_tfjs_model(write_model(str(tmp_path / "b"), dims=(53, 40, 3), acts=("sigmoid", "linear"), seed=3))
    c2 = predict.Classifier(m2)
    assert np.abs(c2.probabilities(rows[10:60]) - forward_f32(m2, rows[10:60])).max() < 1e-4
    clf.close(); c2.close()


@pytest.mark.gpu
def test_classify_feature_rows_where_they_are(tmp_path):
    """Rows of a finished batch are classified on the device; same scores as sending the copied rows through the host entry."""
    from webspeechanalyzer_b200 import Engine, FaConfig, api, synth_speech
    m = predict.load_tfjs_model(write_model(str(tmp_path)))
    clf = predict.Classifier(m)
    sr = 16000
    cfg = FaConfig.default(output_level=13, window_step_ms=15.0)
    with Engine(cfg) as eng:
        for u in range(6):
            eng.submit(u, synth_speech(5 * sr, sr, 5, u), sr)
        eng.run(); eng.sync()
        allp = clf.classify_features(eng)
        rows = eng.result(None).features
        assert allp.shape == (rows.shape[0], 4) and rows.shape[0] > 6
        assert np.array_equal(allp, clf.probabilities(rows), equal_nan=True)
        r3 = eng.result(3)
        p3 = clf.classify_features(eng, 3)
        assert np.array_equal(p3, clf.probabilities(r3.features), equal_nan=True)
        # the app's flow: per segment, the syllable rows vote with sqrt(duration) weights
        voter = predict.SegmentVoter([1])
        calls = api.segment_callbacks(13, 15.0, [], r3)
        k = 0
        for si, _, times, payload in calls:
            res = clf.results(p3[k: k + len(payload)])
            k += len(payload)
            top, conf = voter.segment({1: res}, times)
            assert top in clf.labels and 0 < conf
    with Engine(FaConfig.default(output_level=4)) as eng:
        eng.submit(0, synth_speech(sr, sr, 1, 0), sr)
        eng.run(); eng.sync()
        with pytest.raises(Exception):
            clf.classify_features(eng)
    clf.close()


def test_segment_vote_matches_reference_prediction_js():
    """SegmentVoter against what the reference's own src/prediction.js passed to its callback (executed by oracle/minijs;
    tests/golden/make_ref_js_vote_golden.py): label and confidence bit for bit, including the one-syllable quirk (only the top
    class of the flat list counts), exact ties and zero-duration segments (no callback)."""
    here = os.path.dirname(os.path.abspath(__file__))
    doc = json.load(open(os.path.join(here, "golden", "ref_js_vote.json")))
    n = 0
    for segs in doc["clips"]:
        v = predict.SegmentVoter((1,))
        for s in segs:
            res, st = s["results"], s["seg_time"]
            got = v.segment({1: [res] if len(st) == 1 else res}, st)
            want = s["reference_callback"]
            assert (got is None) == (want is None)
            if want is not None:
                assert got[0] == want[0] and got[1] == want[1], (got, want)
            n += 1
    assert n >= 20
    if os.path.exists("/root/reference/src/prediction.js"):      # build container: execute the reference again, live
        import sys
        sys.path.insert(0, os.path.join(here, "golden"))
        from make_ref_js_vote_golden import reference_votes
        for segs in doc["clips"][:2]:
            live = reference_votes([(s["results"], s["seg_time"]) for s in segs])
            assert live == [s["reference_callback"] for s in segs]


@pytest.mark.gpu
def test_shipped_models_against_float64():
    """The reference's shipped classifiers (dist/nnmodel/{1,2,4..7}/cats_emotion; 4-7 share one weight file) scored by the
    CUDA kernel on real 53-dim rows of the demo WAV, against an independent float64 forward pass
    (tests/golden/make_mlp_golden.py): same arg-max on every row, class scores within 1e-5.  Model 4 (53-512-512-8, 1.2 MB of
    parameters) takes the kernel variant that reads the parameters from L2 instead of shared memory."""
    here = os.path.dirname(os.path.abspath(__file__))
    import sys
    sys.path.insert(0, os.path.join(here, "golden"))
    import npzparts
    z = npzparts.load(os.path.join(here, "golden", "mlp_shipped"))
    info = json.load(open(os.path.join(here, "golden", "mlp_shipped.json")))
    rows = z["rows"]
    assert rows.shape == (info["rows"], 53) and rows.shape[0] >= 30
    for db, mi in info["models"].items():
        n = len(mi["dims"]) - 1
        model = dict(dims=mi["dims"], activations=mi["activations"], kernels=[z[f"m{db}_k{i}"] for i in range(n)],
                     biases=[z[f"m{db}_b{i}"] for i in range(n)], in_min=z[f"m{db}_min"], in_max=z[f"m{db}_max"], labels=mi["labels"])
        clf = predict.Classifier(model)
        p = clf.probabilities(rows)
        want = z[f"m{db}_expected"]
        assert p.shape == want.shape
        assert np.array_equal(p.argmax(axis=1), want.argmax(axis=1)), db
        assert np.abs(p.astype(np.float64) - want).max() <= 1e-5, (db, np.abs(p - want).max())
        assert np.allclose(p.sum(axis=1), 1.0, atol=1e-5)
        res = clf.classify_multiple(rows[:2])
        assert res[0][0]["label"] == mi["labels"][int(want[0].argmax())]
        clf.close()
