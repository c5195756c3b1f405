"""Training of the feature-row classifier (K9, csrc/fa_train.cu; algorithm in DESIGN.md "K9").

CPU: the model writer round-trips through the loader, the numpy restatement of the batch order is a bijection, the options
struct matches the header, host-side rejections, and no CPU fallback.  GPU: SGD and Adam against this file's own float64
trainer of the same algorithm (same start values, order and ranges), determinism and job independence, learning,
fine-tune passthrough, real rows from an Engine and the device-side rejection of non-finite rows."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from test_predict import forward_f32, write_model
from webspeechanalyzer_b200 import _capi, predict
from webspeechanalyzer_b200._capi import FaError

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
M32, M64 = 0xFFFFFFFF, (1 << 64) - 1


# ---- numpy restatement of include/fa_train.h ----------------------------------------------------------------------------
def _mix64(z):
    z = (z + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def perm(n, seed, epoch):
    """Position i -> fa_perm(i, n, seed, epoch) for i in [0, n)."""
    h = 1
    while h < 16 and (1 << (2 * h)) < n:
        h += 1
    mask = np.uint32((1 << h) - 1)
    keys = [np.uint32(_mix64(_mix64(seed & M64) ^ (epoch << 8) ^ r) & M32) for r in range(4)]

    def enc(x):
        lo, hi = x >> np.uint32(h), x & mask
        for k in keys:
            f = hi ^ k
            f ^= f >> np.uint32(16); f *= np.uint32(0x7FEB352D)
            f ^= f >> np.uint32(15); f *= np.uint32(0x846CA68B)
            f ^= f >> np.uint32(16)
            lo, hi = hi, lo ^ (f & mask)
        return (lo << np.uint32(h)) | hi

    with np.errstate(over="ignore"):
        x = enc(np.arange(n, dtype=np.uint32))
        out = x >= n
        while out.any():
            x[out] = enc(x[out])
            out = x >= n
    return x.astype(np.int64)


# ---- float64 trainer of the same algorithm ------------------------------------------------------------------------------
def split(flat, dims):
    Ws, bs, off = [], [], 0
    for a, b in zip(dims[:-1], dims[1:]):
        Ws.append(np.asarray(flat[off: off + a * b], np.float64).reshape(a, b).copy()); off += a * b
        bs.append(np.asarray(flat[off: off + b], np.float64).copy()); off += b
    return Ws, bs


def job_ranges(rows, idx):
    lo, hi = rows[idx].min(axis=0), rows[idx].max(axis=0)
    return lo, np.where(hi == lo, lo + 1.0, hi)


def train_f64(rows, labels, dims, acts, flat, lo, hi, idx, seed, epochs, batch, optimizer, lr):
    """Returns (weights, biases, [(loss, accuracy)] per epoch, per-step gradients)."""
    Ws, bs = split(flat, dims)
    x_all = ((rows - lo) / (hi - lo)).astype(np.float32).astype(np.float64)
    ms = [np.zeros_like(w) for w in Ws + bs]
    vs = [np.zeros_like(w) for w in Ws + bs]
    n, t, hist, grads_log = len(idx), 0, [], []
    for e in range(epochs):
        order = idx[perm(n, seed, e)]
        loss, hits = 0.0, 0
        for s0 in range(0, n, batch):
            rb = order[s0: s0 + batch]
            bc = len(rb)
            a = [x_all[rb]]
            for l in range(len(Ws)):
                z = a[-1] @ Ws[l] + bs[l]
                if acts[l] == 1:
                    z = np.maximum(z, 0)
                elif acts[l] == 2:
                    z = 1 / (1 + np.exp(-z))
                elif acts[l] == 3:
                    z = np.exp(z - z.max(axis=1, keepdims=True))
                    z /= z.sum(axis=1, keepdims=True)
                a.append(z)
            p, y = a[-1], labels[rb]
            loss += float(-np.log(np.maximum(p[np.arange(bc), y], 1e-7)).sum())
            hits += int((p.argmax(axis=1) == y).sum())
            dz = p.copy()
            dz[np.arange(bc), y] -= 1
            dz /= bc
            gW, gb = [None] * len(Ws), [None] * len(Ws)
            for l in range(len(Ws) - 1, -1, -1):
                gW[l], gb[l] = a[l].T @ dz, dz.sum(axis=0)
                if l:
                    da = dz @ Ws[l].T
                    dz = da * (a[l] > 0) if acts[l - 1] == 1 else da * a[l] * (1 - a[l]) if acts[l - 1] == 2 else da
            t += 1
            grads = gW + gb
            grads_log.append(grads)
            for i, (w, g) in enumerate(zip(Ws + bs, grads)):
                if optimizer == "sgd":
                    w -= lr * g
                else:
                    ms[i] = 0.9 * ms[i] + 0.1 * g
                    vs[i] = 0.999 * vs[i] + 0.001 * g * g
                    w -= lr * (ms[i] / (1 - 0.9 ** t)) / (np.sqrt(vs[i] / (1 - 0.999 ** t)) + 1e-7)
        hist.append((loss / n, hits / n))
    return Ws, bs, hist, grads_log


def four_class(n, seed, spread=1.0, d=53):
    """Seeded 4-class rows: class centres in a 53-dim space with per-column scales and offsets; column 5 is constant."""
    rng = np.random.default_rng(seed)
    centres = rng.normal(0, 1, (4, d))
    y = rng.integers(0, 4, n).astype(np.int32)
    x = centres[y] + spread * rng.normal(0, 1, (n, d))
    x = x * rng.uniform(0.5, 200, d) + rng.uniform(-50, 50, d)
    x[:, 5] = 3.25
    return x, y


def model_of(m):
    return {k: m[k] for k in ("dims", "activations", "kernels", "biases", "in_min", "in_max", "labels")}


# ---- CPU --------------------------------------------------------------------------------------------------------------
def assert_same_model(a, b):
    assert list(a["dims"]) == list(b["dims"]) and list(a["activations"]) == list(b["activations"])
    assert list(a["labels"]) == list(b["labels"])
    for x, y in zip(a["kernels"] + a["biases"], b["kernels"] + b["biases"]):
        assert x.dtype == y.dtype == np.float32 and x.shape == y.shape and x.tobytes() == y.tobytes()
    assert np.asarray(a["in_min"]).tobytes() == np.asarray(b["in_min"]).tobytes()
    assert np.asarray(a["in_max"]).tobytes() == np.asarray(b["in_max"]).tobytes()


def test_save_then_load_returns_the_same_model(tmp_path):
    rng = np.random.default_rng(7)
    dims = [53, 40, 12, 3]
    m = dict(dims=dims, activations=[2, 0, 3], labels=["sad", "angry", "calm"],
             kernels=[rng.normal(0, 1, (a, b)).astype(np.float32) for a, b in zip(dims[:-1], dims[1:])],
             biases=[rng.normal(0, 1, b).astype(np.float32) for b in dims[1:]],
             in_min=rng.normal(0, 100, 53), in_max=rng.normal(0, 100, 53) + 1000)
    m["kernels"][0][3, 4] = -0.0
    d = predict.save_tfjs_model(m, str(tmp_path / "m"))
    assert sorted(os.listdir(d)) == ["model.json", "model.weights.bin", "model_meta.json"]
    meta = json.load(open(os.path.join(d, "model_meta.json")))
    assert meta["isNormalized"] is True and meta["inputUnits"] == [53] and meta["outputUnits"] == 3
    assert meta["outputs"]["label"]["uniqueValues"] == ["sad", "angry", "calm"]
    doc = json.load(open(os.path.join(d, "model.json")))
    assert doc["weightsManifest"][0]["paths"] == ["./model.weights.bin"]
    assert_same_model(m, predict.load_tfjs_model(d))


def test_fixture_model_survives_load_save_load(tmp_path):
    a = predict.load_tfjs_model(write_model(str(tmp_path / "a")))
    b = predict.load_tfjs_model(predict.save_tfjs_model(a, str(tmp_path / "b")))
    assert_same_model(a, b)
    c = predict.load_tfjs_model(write_model(str(tmp_path / "c"), dims=(53, 40, 3), acts=("sigmoid", "softmax"), seed=3))
    assert_same_model(c, predict.load_tfjs_model(predict.save_tfjs_model(c, str(tmp_path / "d"))))


@pytest.mark.parametrize("n", [1, 2, 31, 32, 33, 1000, 74249])
def test_batch_order_is_a_bijection(n):
    p = perm(n, 5, 0)
    assert np.array_equal(np.sort(p), np.arange(n))
    if n >= 31:
        assert not np.array_equal(p, perm(n, 5, 1)) and not np.array_equal(p, perm(n, 6, 0))
        assert not np.array_equal(p, np.arange(n))


def test_numpy_batch_order_equals_the_header(tmp_path):
    """The restatement above against include/fa_train.h itself, compiled for the host."""
    src = tmp_path / "perm.c"
    src.write_text('#include <stdio.h>\n#include <stdlib.h>\n#include "fa_train.h"\nint main(int c, char** v) {\n'
                   '  unsigned n = (unsigned)atol(v[1]); unsigned long long s = strtoull(v[2], 0, 10); unsigned e = (unsigned)atol(v[3]);\n'
                   '  for (unsigned i = 0; i < n; i++) printf("%u\\n", fa_perm(i, n, s, e));\n  return 0;\n}\n')
    exe = str(tmp_path / "perm")
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), "-o", exe, str(src)])
    for n, seed, epoch in ((1, 0, 0), (33, 7, 2), (1000, 2**63 + 5, 11), (74249, 3, 999)):
        got = np.array(subprocess.check_output([exe, str(n), str(seed), str(epoch)], text=True).split(), np.int64)
        assert np.array_equal(got, perm(n, seed, epoch)), (n, seed, epoch)


def test_options_struct_matches_the_header(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "fa_b200.h"\nint main(void) {\n'
                   '  printf("%zu %zu %zu %zu %zu\\n", sizeof(fa_train_opts), offsetof(fa_train_opts, learning_rate),\n'
                   '         offsetof(fa_train_opts, optimizer), offsetof(fa_train_opts, epochs), offsetof(fa_train_opts, batch_size));\n'
                   '  return 0;\n}\n')
    exe = str(tmp_path / "layout")
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), "-o", exe, str(src)])
    got = [int(x) for x in subprocess.check_output([exe], text=True).split()]
    T = _capi.FaTrainOpts
    want = [C.sizeof(T)] + [getattr(T, f).offset for f in ("learning_rate", "optimizer", "epochs", "batch_size")]
    assert got == want and [f for f, _ in T._fields_] == ["learning_rate", "optimizer", "epochs", "batch_size"]


def expect_invalid(match, *args, **kw):
    with pytest.raises(FaError) as e:
        predict.train(*args, **kw)
    assert e.value.status == _capi.FA_ERR_INVALID_ARG and match in e.value.message, e.value.message


def test_rejections_on_the_host(tmp_path):
    """Checked before any device is touched, so they hold on every machine."""
    x, y = four_class(100, 1)
    names = ["a", "b", "c", "d"]
    bad = y.copy(); bad[17] = 4
    expect_invalid("label 4 of row 17 is outside [0, 4)", x, bad, names, epochs=1)
    bad[17] = -1
    expect_invalid("label -1 of row 17", x, bad, names, epochs=1)
    expect_invalid("row index 100 at position 3", x, y, names, jobs=[[0, 1, 2, 100]], epochs=1)
    expect_invalid("row index -1", x, y, names, jobs=[[-1]], epochs=1)
    expect_invalid("job 1 is empty", x, y, names, jobs=[[0, 1], []], epochs=1)
    expect_invalid("batch_size", x, y, names, batch_size=0, epochs=1)
    expect_invalid("epochs must be >= 0", x, y, names, epochs=-1)
    init = predict.load_tfjs_model(write_model(str(tmp_path / "a"), acts=("relu", "relu", "relu", "relu")))
    expect_invalid("output activation must be softmax", x, y, names, init=init, epochs=1)
    init = predict.load_tfjs_model(write_model(str(tmp_path / "b"), acts=("softmax", "relu", "relu", "softmax")))
    expect_invalid("hidden layer 0", x, y, names, init=init, epochs=1)


NO_DEVICE_CHECK = """
import numpy as np
from webspeechanalyzer_b200 import _capi, predict
x = np.random.default_rng(0).normal(size=(40, 53))
try:
    predict.train(x, np.arange(40) % 4, list("abcd"), epochs=1)
    raise AssertionError("train() without a device")
except _capi.FaError as e:
    assert e.status == _capi.FA_ERR_NO_DEVICE, e
"""


def test_no_cpu_fallback():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    subprocess.run([sys.executable, "-c", NO_DEVICE_CHECK], cwd=ROOT, env=env, check=True)


# ---- GPU --------------------------------------------------------------------------------------------------------------
def layer_close(got, Ws, bs, tol=1e-4, exempt=None):
    """Every parameter within tol x the layer's largest |w| of the float64 reference (exempt: masks of skipped entries)."""
    nl = len(Ws)
    for l in range(nl):
        scale = max(np.abs(Ws[l]).max(), np.abs(bs[l]).max())
        for i, (g, r) in enumerate(((got["kernels"][l], Ws[l]), (got["biases"][l], bs[l]))):
            d = np.abs(g.astype(np.float64) - r)
            if exempt is not None:
                d = np.where(exempt[l + i * nl], 0, d)
            assert d.max() <= tol * scale, (l, i, d.max(), scale)


@pytest.mark.gpu
def test_sgd_matches_float64():
    x, y = four_class(2000, 11)
    names = ["N", "A", "S", "H"]
    m = predict.train(x, y, names, hidden=(256, 64, 16), optimizer="sgd", learning_rate=0.1, epochs=3, batch_size=32, seed=3)
    dims, acts = [53, 256, 64, 16, 4], [1, 1, 1, 3]
    lo, hi = job_ranges(x, np.arange(2000))
    assert np.array_equal(m["in_min"], lo) and np.array_equal(m["in_max"], hi) and m["in_max"][5] == 4.25
    Ws, bs, hist, _ = train_f64(x, y, dims, acts, predict.glorot_params(dims, 3), lo, hi, np.arange(2000), 3, 3, 32, "sgd", 0.1)
    layer_close(m, Ws, bs)
    ref = np.array(hist)
    assert np.all(np.abs(m["history"]["loss"] - ref[:, 0]) <= 1e-5 * ref[:, 0])
    assert np.all(np.abs(m["history"]["accuracy"] - ref[:, 1]) <= 2 / 2000)
    assert m["history"]["loss"][-1] < m["history"]["loss"][0]


@pytest.mark.gpu
def test_adam_matches_float64():
    x, y = four_class(2000, 12)
    names = ["N", "A", "S", "H"]
    dims, acts = [53, 256, 64, 16, 4], [1, 1, 1, 3]
    idx = np.arange(160)                                    # one epoch = 5 steps of 32
    lo, hi = job_ranges(x, idx)
    m = predict.train(x, y, names, optimizer="adam", learning_rate=1e-3, epochs=1, jobs=[idx], seed=[4])[0]
    Ws, bs, _, grads = train_f64(x, y, dims, acts, predict.glorot_params(dims, 4), lo, hi, idx, 4, 1, 32, "adam", 1e-3)
    assert len(grads) == 5
    nl = len(Ws)
    exempt = [np.zeros(g.shape, bool) for g in grads[0]]
    for gs in grads:                   # a near-zero gradient's sign decides +-lr in m / sqrt(v)
        for l in range(nl):
            big = max(np.abs(gs[l]).max(), np.abs(gs[l + nl]).max())
            exempt[l] |= np.abs(gs[l]) < 1e-6 * big
            exempt[l + nl] |= np.abs(gs[l + nl]) < 1e-6 * big
    layer_close(m, Ws, bs, exempt=exempt)
    m5 = predict.train(x, y, names, optimizer="adam", learning_rate=1e-3, epochs=5, seed=5)
    _, _, hist, _ = train_f64(x, y, dims, acts, predict.glorot_params(dims, 5), *job_ranges(x, np.arange(2000)),
                              np.arange(2000), 5, 5, 32, "adam", 1e-3)
    ref = np.array(hist)[:, 0]
    assert np.all(np.abs(m5["history"]["loss"] - ref) <= 1e-3 * ref)


@pytest.mark.gpu
def test_runs_are_deterministic_and_jobs_independent():
    x, y = four_class(1500, 13)
    names = ["N", "A", "S", "H"]
    rng = np.random.default_rng(2)
    jobs = [rng.choice(1500, size=int(rng.integers(40, 700)), replace=bool(j % 2)) for j in range(9)]
    seeds = list(range(100, 109))
    kw = dict(hidden=(64, 16), optimizer="adam", epochs=3, batch_size=24)
    a = predict.train(x, y, names, jobs=jobs, seed=seeds, **kw)
    b = predict.train(x, y, names, jobs=jobs, seed=seeds, **kw)
    for ma, mb in zip(a, b):
        assert_same_model(ma, mb)
        assert ma["history"]["loss"].tobytes() == mb["history"]["loss"].tobytes()
    for j in (0, 4, 8):
        alone = predict.train(x, y, names, jobs=[jobs[j]], seed=[seeds[j]], **kw)[0]
        assert_same_model(a[j], alone)
        assert a[j]["history"]["loss"].tobytes() == alone["history"]["loss"].tobytes()
        assert a[j]["history"]["accuracy"].tobytes() == alone["history"]["accuracy"].tobytes()
    assert a[0]["kernels"][0].tobytes() != a[1]["kernels"][0].tobytes()


@pytest.mark.gpu
def test_learns_separable_classes(tmp_path):
    x, y = four_class(2000, 14, spread=0.3)
    names = ["N", "A", "S", "H"]
    m = predict.train(x[:1600], y[:1600], names, seed=1)
    assert len(m["history"]["loss"]) == 32 and m["history"]["accuracy"][-1] >= 0.95
    back = predict.load_tfjs_model(predict.save_tfjs_model(m, str(tmp_path / "m")))
    assert_same_model(model_of(m), back)
    clf = predict.Classifier(back)
    p = clf.probabilities(x[1600:])
    assert (p.argmax(axis=1) == y[1600:]).mean() >= 0.95
    assert np.abs(p - forward_f32(back, x[1600:])).max() <= 1e-5
    clf.close()


@pytest.mark.gpu
def test_zero_learning_rate_passes_the_shipped_model_through():
    sys.path.insert(0, GOLDEN)
    import npzparts
    z = npzparts.load(os.path.join(GOLDEN, "mlp_shipped"))
    info = json.load(open(os.path.join(GOLDEN, "mlp_shipped.json")))
    mi = info["models"]["1"]
    n = len(mi["dims"]) - 1
    init = dict(dims=mi["dims"], activations=mi["activations"], kernels=[z[f"m1_k{i}"] for i in range(n)],
                biases=[z[f"m1_b{i}"] for i in range(n)], in_min=z["m1_min"], in_max=z["m1_max"], labels=mi["labels"])
    rows = z["rows"]
    y = z["m1_expected"].argmax(axis=1).astype(np.int32)
    for opt in ("sgd", "adam"):
        m = predict.train(rows, y, mi["labels"], optimizer=opt, learning_rate=0.0, epochs=2, batch_size=8, init=init)
        assert_same_model(model_of(m), dict(init, kernels=[np.asarray(k, np.float32) for k in init["kernels"]],
                                            biases=[np.asarray(b, np.float32) for b in init["biases"]],
                                            in_min=np.asarray(init["in_min"], np.float64), in_max=np.asarray(init["in_max"], np.float64)))
        assert np.all(np.isfinite(m["history"]["loss"]))


@pytest.mark.gpu
def test_trains_on_engine_rows():
    from webspeechanalyzer_b200 import Engine, FaConfig, synth_speech
    sr = 16000
    n_utt = 24                                              # ~0.7 syllable rows per second of this speech: ~100 rows
    utt_labels = [u % 3 for u in range(n_utt)]
    with Engine(FaConfig.default(output_level=13, window_step_ms=15.0)) as eng:
        for u in range(n_utt):
            eng.submit(u, synth_speech(6 * sr, sr, 20 + (u % 3), u), sr)
        eng.run(); eng.sync()
        rows = eng.feature_table()
        labels = predict.row_labels(eng, utt_labels)
        assert labels.shape == (rows.shape[0],) and rows.shape[0] > 30
        assert np.array_equal(labels[:eng.counts(0)["feature_rows"]], np.zeros(eng.counts(0)["feature_rows"]))
        ok = np.isfinite(rows).all(axis=1)
        m = predict.train(rows[ok], labels[ok], ["x", "y", "z"], hidden=(64, 16), epochs=30, batch_size=16, seed=2)
        assert m["history"]["loss"][-1] < m["history"]["loss"][0]
        clf = predict.Classifier(m)
        p = clf.classify_features(eng)
        assert p.shape == (rows.shape[0], 3)
        assert np.allclose(p[ok].sum(axis=1), 1, atol=1e-5)
        assert np.array_equal(p, clf.probabilities(rows), equal_nan=True)
        clf.close()
        with pytest.raises(ValueError):
            predict.row_labels(eng, utt_labels[:-1])


@pytest.mark.gpu
def test_rejects_non_finite_selected_rows():
    x, y = four_class(100, 15)
    names = ["a", "b", "c", "d"]
    x[37, 9] = np.nan
    x[61, 2] = np.inf
    expect_invalid("row 37 has a non-finite value", x, y, names, epochs=1)
    expect_invalid("row 61 has a non-finite value", x, y, names, jobs=[np.arange(40, 100)], epochs=1)
    m = predict.train(x, y, names, jobs=[np.arange(0, 30), np.arange(70, 100)], epochs=1, hidden=(8,))
    assert len(m) == 2 and all(np.isfinite(k["kernels"][0]).all() for k in m)
