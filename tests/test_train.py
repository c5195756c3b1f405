"""Training of the feature-row classifier (K9, csrc/fa_train.cu; algorithm in DESIGN.md "K9").

CPU: the model writer round-trips through the loader, the numpy restatement of the batch order is a bijection, the options
struct matches the header, the launch geometry fits every accepted input, host-side rejections, and no CPU fallback.
GPU: SGD and Adam against this file's own float64 trainer of the same algorithm (same start values, order and ranges) --
on the default shape and on a table of cases that takes every branch of the kernel -- determinism and job independence,
learning, fine-tune passthrough, real rows from an Engine and the device-side rejection of non-finite rows."""
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


def four_class(n, seed, spread=1.0, d=53, k=4):
    """Seeded rows of k classes (4 by default): class centres in a d-dim space with per-column scales and offsets; column 5
    (if there is one) is constant."""
    rng = np.random.default_rng(seed)
    centres = rng.normal(0, 1, (k, d))
    y = rng.integers(0, k, n).astype(np.int32)
    x = centres[y] + spread * rng.normal(0, 1, (n, d))
    x = x * rng.uniform(0.5, 200, d) + rng.uniform(-50, 50, d)
    if d > 5:
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


GEOMETRY_C = r"""#include <stdio.h>
#include <stdlib.h>
#include "fa_train.h"
int main(int argc, char** argv) {   /* batch smem_optin dims[0] .. dims[n_layers] */
  int dims[FA_MLP_MAX_LAYERS + 1], n_layers = argc - 4;
  for (int l = 0; l <= n_layers; l++) dims[l] = atoi(argv[3 + l]);
  fa_train_geom g;
  int rc = fa_train_geometry(dims, n_layers, atoi(argv[1]), 200 * 1024, atoll(argv[2]), &g);
  printf("%d %lld %lld %lld %lld %lld %lld %d %lld", rc, (long long)g.bpad, (long long)g.n_params, (long long)g.n_act,
         (long long)g.act_off, (long long)g.area_bytes, (long long)g.area_smem_off, g.area_in_smem, (long long)g.smem_bytes);
  for (int l = 0; l <= n_layers; l++) printf(" %lld", (long long)g.a_off[l]);
  for (int l = 0; l < n_layers; l++) printf(" %lld %lld", (long long)g.w_off[l], (long long)g.b_off[l]);
  printf("\n");
  return 0;
}
"""
SMEM_OPTIN = 227 * 1024 - 16      # a B200 block's opt-in shared memory minus fa_train_kernel's 16 bytes of static shared memory


def geometry_py(dims, batch, cap=200 * 1024):
    """DESIGN.md "K9" / include/fa_train.h restated: red + rng, then the batch area (per-row tables: 8 + 3 x 4 bytes a
    row; activations) in shared memory when the launch stays under `cap`, else in per-job global scratch."""
    bpad = -(-batch // 8) * 8
    a_off = [bpad * sum(dims[:l]) for l in range(len(dims))]
    wb, off = [], 0
    for a, b in zip(dims[:-1], dims[1:]):
        wb += [off, off + a * b]
        off += a * b + b
    n_act = bpad * sum(dims)
    act_off = 20 * bpad
    area = -(-(act_off + 4 * n_act) // 16) * 16
    area_smem_off = 8 * (2 * 512 + 2 * dims[0])
    in_smem = int(area_smem_off + area <= cap)
    return [0, bpad, off, n_act, act_off, area, area_smem_off, in_smem, area_smem_off + (area if in_smem else 0)] + a_off + wb


@pytest.mark.parametrize("dims, batch, in_smem", [
    ((53, 256, 64, 16, 4), 32, 1),          # the default shape: 59 984 B of shared memory
    ((53, 256, 64, 16, 4), 256, 0),         # activations past the 200 KB cap
    ((53, 48, 24, 12, 5), 20, 1),           # padding rows
    ((1, 4, 2), 1, 1),
    ((53, 8, 4), 11170, 0),                 # per-row tables in shared memory would pass 227 KB here
    ((53, 8, 4), 12000, 0),
    ((53, 8, 4), 65536, 0),                 # the largest batch
    ((3200, 64, 4), 8700, 0),               # the widest input: 50 KB of ranges
    ((3200,) * 9, 65536, 0),                # the largest model the host accepts
], ids=lambda v: "-".join(map(str, v)) if isinstance(v, tuple) else str(v))
def test_launch_geometry_fits_every_accepted_input(tmp_path, dims, batch, in_smem):
    """fa_train_geometry (include/fa_train.h, what fa_mlp_train launches with): every input the host accepts fits the
    block's shared memory, its activation offsets fit the kernel's 32-bit indexing, and the layout is the restated one."""
    src = tmp_path / "geom.c"
    src.write_text(GEOMETRY_C)
    exe = str(tmp_path / "geom")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", exe, str(src)])

    def run(optin):
        return [int(v) for v in subprocess.check_output([exe, str(batch), str(optin), *map(str, dims)], text=True).split()]
    got = run(SMEM_OPTIN)
    assert got == geometry_py(dims, batch)
    rc, n_act, in_smem_got, smem = got[0], got[3], got[7], got[8]
    assert rc == 0 and in_smem_got == in_smem and smem <= SMEM_OPTIN and n_act <= 2**31 - 1
    assert run(smem)[0] == 0 and run(smem - 1)[0] == -1
    if dims == (53, 256, 64, 16, 4) and batch == 32:
        assert smem == 59984


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
    # FA_MLP_MAX_UNITS: a wider layer, or a wider input, would train and then not load into Classifier
    expect_invalid("dims[1] must be in [1, 3200]", x, y, names, hidden=(3201,), epochs=1)
    expect_invalid("dims[2] must be in [1, 3200]", x, y, names, hidden=(16, 4000), epochs=1)
    wide, wy = four_class(20, 2, d=3201)
    expect_invalid("dims[0] must be in [1, 3200]", wide, wy, names, hidden=(8,), epochs=1)


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


def adam_exempt(grads):
    """Masks of the parameters whose gradient was near zero at some step: its sign decides +-lr in m / sqrt(v)."""
    nl = len(grads[0]) // 2
    exempt = [np.zeros(g.shape, bool) for g in grads[0]]
    for gs in grads:
        for l in range(nl):
            big = max(np.abs(gs[l]).max(), np.abs(gs[l + nl]).max())
            exempt[l] |= np.abs(gs[l]) < 1e-6 * big
            exempt[l + nl] |= np.abs(gs[l + nl]) < 1e-6 * big
    return exempt


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
    layer_close(m, Ws, bs, exempt=adam_exempt(grads))
    m5 = predict.train(x, y, names, optimizer="adam", learning_rate=1e-3, epochs=5, seed=5)
    _, _, hist, _ = train_f64(x, y, dims, acts, predict.glorot_params(dims, 5), *job_ranges(x, np.arange(2000)),
                              np.arange(2000), 5, 5, 32, "adam", 1e-3)
    ref = np.array(hist)[:, 0]
    assert np.all(np.abs(m5["history"]["loss"] - ref) <= 1e-3 * ref)


# ---- every path of the kernel against the float64 trainer, each run a few dozen steps at most -------------------------
NAMES4 = ["N", "A", "S", "H"]


def flat_of(m):
    return np.concatenate([np.asarray(a, np.float32).ravel() for k, b in zip(m["kernels"], m["biases"]) for a in (k, b)])


def train_and_check(x, y, names, jobs, seeds, hidden=(), acts="relu", optimizer="sgd", lr=0.1, epochs=1, batch=32, init=None):
    """predict.train on `jobs`, then every job against train_f64 from the same start values, order and ranges: parameters
    within 1e-4 of the layer's largest |w| (Adam: but for near-zero gradients), per-epoch loss within 1e-5 (SGD) or 1e-3
    (Adam) relative, accuracy within 2 rows, ranges bit-equal; and K7 scores every model within 1e-5 of forward_f32."""
    models = predict.train(x, y, names, hidden=hidden, activations=acts, optimizer=optimizer, learning_rate=lr,
                           epochs=epochs, batch_size=batch, jobs=jobs, seed=seeds, init=init)
    for m, idx, seed in zip(models, jobs, seeds):
        idx = np.asarray(idx)
        if init is None:
            lo, hi = job_ranges(x, idx)
            flat = predict.glorot_params(m["dims"], seed)
        else:
            lo, hi = np.asarray(init["in_min"], np.float64), np.asarray(init["in_max"], np.float64)
            flat = flat_of(init)
        assert m["in_min"].tobytes() == lo.tobytes() and m["in_max"].tobytes() == hi.tobytes()
        Ws, bs, hist, grads = train_f64(x, y, m["dims"], m["activations"], flat, lo, hi, idx, seed, epochs, batch, optimizer, lr)
        layer_close(m, Ws, bs, exempt=adam_exempt(grads) if optimizer == "adam" else None)
        ref = np.array(hist)
        rel = 1e-5 if optimizer == "sgd" else 1e-3
        assert np.all(np.abs(m["history"]["loss"] - ref[:, 0]) <= rel * ref[:, 0]), (m["history"]["loss"], ref[:, 0])
        assert np.all(np.abs(m["history"]["accuracy"] - ref[:, 1]) <= 2 / len(idx))
        rows = x[idx[:1024]]
        clf = predict.Classifier(m)
        assert np.abs(clf.probabilities(rows) - forward_f32(m, rows)).max() <= 1e-5
        clf.close()
    return models


def case_sigmoid():
    x, y = four_class(1000, 21)
    for opt, lr in (("sgd", 0.5), ("adam", 1e-3)):
        train_and_check(x, y, NAMES4, [np.arange(1000)], [7], hidden=(64, 16), acts="sigmoid", optimizer=opt, lr=lr)


def case_mixed():
    """linear backward, 5 classes, 4 padding rows per batch of 20, a last batch of 17"""
    x, y = four_class(517, 22, k=5)
    train_and_check(x, y, list("abcde"), [np.arange(517)], [8], hidden=(48, 24, 12), acts=["linear", "sigmoid", "relu"],
                    lr=0.2, batch=20)


def case_no_hidden():
    """one layer (no delta phase), one padding row per batch of 7"""
    x, y = four_class(300, 23, k=3)
    train_and_check(x, y, list("abc"), [np.arange(300)], [9], lr=0.5, batch=7)


def case_deep():
    x, y = four_class(320, 24)
    train_and_check(x, y, NAMES4, [np.arange(320)], [10], hidden=(32,) * 7, acts=["relu", "sigmoid"] * 3 + ["relu"],
                    lr=0.5, batch=16)


def case_wide():
    """widths above the 512 threads of a job and not a multiple of 32, 2 classes"""
    x, y = four_class(200, 25, k=2)
    train_and_check(x, y, ["x", "y"], [np.arange(200)], [11], hidden=(600, 37), lr=0.1, batch=8)


def case_inputs():
    """the range reduction over 1, 2 and 3 chunks of 512 columns, constant columns in the first and the last chunk"""
    x, y = four_class(300, 26, d=1, k=2)
    train_and_check(x, y, ["x", "y"], [np.arange(300)], [12], hidden=(4,), lr=0.5)
    for d in (600, 1030):
        x, y = four_class(400, 27, d=d)
        x[:, d - 1] = -7.5
        train_and_check(x, y, NAMES4, [np.arange(13, 269)], [13], hidden=(16,), lr=0.1)


def case_batch_edges():
    x, y = four_class(200, 28)
    train_and_check(x, y, NAMES4, [np.arange(40)], [14], hidden=(16,), lr=0.1, batch=1)
    train_and_check(x, y, NAMES4, [np.arange(100, 145)], [15], hidden=(16,), optimizer="adam", lr=1e-3, epochs=3, batch=64)


def case_global_scratch():
    """the default shape at batch 256: per-row tables and activations in per-job slices of global scratch"""
    x, y = four_class(1500, 29)
    rng = np.random.default_rng(3)
    jobs = [rng.choice(1500, 300, replace=False), rng.choice(1500, 700, replace=True), np.arange(200, 720)]
    seeds = [31, 32, 33]
    together = train_and_check(x, y, NAMES4, jobs, seeds, hidden=(256, 64, 16), lr=0.1, epochs=2, batch=256)
    for j in range(3):
        alone = predict.train(x, y, NAMES4, hidden=(256, 64, 16), optimizer="sgd", learning_rate=0.1, epochs=2,
                              batch_size=256, jobs=[jobs[j]], seed=[seeds[j]])[0]
        assert_same_model(model_of(together[j]), model_of(alone))
        assert together[j]["history"]["loss"].tobytes() == alone["history"]["loss"].tobytes()


def case_big_batch():
    """batches whose per-row tables alone exceed a block's shared memory, up to the largest batch accepted"""
    x, y = four_class(66536, 30)
    train_and_check(x, y, NAMES4, [np.arange(30000)], [16], hidden=(8,), lr=0.5, batch=12000)
    train_and_check(x, y, NAMES4, [np.arange(66536)], [17], hidden=(8,), lr=0.5, batch=65536)


def case_fine_tune():
    """shipped model 1 as the start, its ranges as given, and rows outside them (normalised below 0 and above 1)"""
    sys.path.insert(0, GOLDEN)
    import npzparts
    z = npzparts.load(os.path.join(GOLDEN, "mlp_shipped"))
    mi = json.load(open(os.path.join(GOLDEN, "mlp_shipped.json")))["models"]["1"]
    n = len(mi["dims"]) - 1
    init = dict(dims=mi["dims"], activations=mi["activations"], kernels=[z[f"m1_k{i}"] for i in range(n)],
                biases=[z[f"m1_b{i}"] for i in range(n)], in_min=z["m1_min"], in_max=z["m1_max"], labels=mi["labels"])
    lo, hi = np.asarray(z["m1_min"], np.float64), np.asarray(z["m1_max"], np.float64)
    rng = np.random.default_rng(4)
    out = np.array(z["rows"][:25], np.float64)
    up, down = np.split(rng.choice(53, 20, replace=False), 2)
    out[:, up] = hi[up] + (hi - lo)[up] * rng.uniform(0.1, 0.5, (25, 10))
    out[:, down] = lo[down] - (hi - lo)[down] * rng.uniform(0.1, 0.5, (25, 10))
    x = np.vstack([z["rows"], out])
    y = rng.integers(0, 4, x.shape[0]).astype(np.int32)
    for opt, lr in (("sgd", 0.05), ("adam", 1e-3)):
        train_and_check(x, y, mi["labels"], [np.arange(x.shape[0])], [18], optimizer=opt, lr=lr, epochs=2, batch=8, init=init)


def case_jobs():
    """repeated and disjoint row lists of different sizes and seeds; Adam's bias correction runs on across epochs"""
    x, y = four_class(600, 31)
    rng = np.random.default_rng(5)
    p = rng.permutation(600)
    jobs = [rng.choice(600, 96, replace=True), p[:40], p[40:110], np.repeat(p[110:129], 3)]
    train_and_check(x, y, NAMES4, jobs, [41, 42, 43, 44], hidden=(64, 16), optimizer="adam", lr=1e-3, epochs=3)


def case_zero_epochs():
    x, y = four_class(300, 32)
    idx = np.arange(50, 250)
    lo, hi = job_ranges(x, idx)
    for opt in ("sgd", "adam"):
        m = predict.train(x, y, NAMES4, hidden=(64, 16), optimizer=opt, epochs=0, jobs=[idx], seed=[19])[0]
        assert flat_of(m).tobytes() == predict.glorot_params(m["dims"], 19).tobytes()
        assert m["in_min"].tobytes() == lo.tobytes() and m["in_max"].tobytes() == hi.tobytes()
        assert m["history"]["loss"].shape == m["history"]["accuracy"].shape == (0,)


def case_width_limit():
    """FA_MLP_MAX_UNITS: K9's widest layer (activations in global scratch) loads into K7 (parameters read from global
    memory, activations at its 200 KB cap); one unit more is refused by K7 (and by K9 on the host)"""
    x, y = four_class(64, 33)
    m = train_and_check(x, y, NAMES4, [np.arange(64)], [20], hidden=(3200,), lr=0.1)[0]
    wider = dict(model_of(m), dims=[53, 3201, 4], kernels=[np.zeros((53, 3201), np.float32), np.zeros((3201, 4), np.float32)],
                 biases=[np.zeros(3201, np.float32), np.zeros(4, np.float32)])
    with pytest.raises(FaError) as e:
        predict.Classifier(wider)
    assert e.value.status == _capi.FA_ERR_UNSUPPORTED


TRAIN_CASES = {f.__name__[5:]: f for f in (case_sigmoid, case_mixed, case_no_hidden, case_deep, case_wide, case_inputs,
                                           case_batch_edges, case_global_scratch, case_big_batch, case_fine_tune,
                                           case_jobs, case_zero_epochs, case_width_limit)}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(TRAIN_CASES))
def test_kernel_paths_match_float64(case):
    TRAIN_CASES[case]()


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
