"""Emotion / label prediction on the 53-dim rows, the way the web app does it (SURVEY.md 8(f) rank 3).

    reference                                                          here
    ml5.neuralNetwork(...).load(model.json, model_meta.json, weights)  load_tfjs_model(dir)  (tf.js layers format)
    nn.classifyMultiple(rows, cb)   src/neuralmodel.js:540-585          Classifier.classify_multiple(rows)
    nn.train(...) + nn.save()       src/neuralmodel.js:163-403          train(rows, labels, ...) + save_tfjs_model(model, dir)
    predict_by_multiple_syllables / nn_prediction / seg_confidence_sort  SegmentVoter
                                    src/prediction.js:47-169

The forward pass runs on the GPU (csrc/fa_mlp.cu behind fa_mlp_* of include/fa_b200.h), and so does training (csrc/fa_train.cu
behind fa_mlp_train; the algorithm is defined in DESIGN.md "K9"); there is no CPU path.
Classifier.classify_features(engine) classifies the rows of a finished batch where they are -- in HBM.
Model files are read at run time from a directory the caller names (e.g. dist/nnmodel/1/cats_emotion of the web app);
nothing of the reference's models is stored in this repository."""
from __future__ import annotations

import ctypes as C
import json
import math
import os

import numpy as np

from . import _capi
from ._capi import FaError

ACTIVATIONS = {"linear": 0, "relu": 1, "sigmoid": 2, "softmax": 3}
ACTIVATION_NAMES = {v: k for k, v in ACTIVATIONS.items()}
OPTIMIZERS = {"sgd": 0, "adam": 1}
# learning rate when the caller names none: ml5's classification SGD rate, tf.js's Adam default (INTEGRATION.md section 3)
DEFAULT_LEARNING_RATE = {"sgd": 0.2, "adam": 0.001}


def load_tfjs_model(model_dir: str, model_json: str = "model.json", meta_json: str = "model_meta.json") -> dict:
    """tf.js layers-model (Sequential of Dense) + ml5 meta -> dict(dims, activations, kernels, biases, in_min, in_max, labels)."""
    with open(os.path.join(model_dir, model_json)) as f:
        doc = json.load(f)
    with open(os.path.join(model_dir, meta_json)) as f:
        meta = json.load(f)
    topo = doc["modelTopology"]
    layers = (topo.get("config") or topo["model_config"]["config"])["layers"]
    dense = [l for l in layers if l["class_name"] == "Dense"]
    if len(dense) != len(layers):
        raise ValueError("only Sequential models of Dense layers are supported")
    # weights: manifest order, float32 little-endian, concatenated over the listed files
    blobs, specs = b"", []
    for group in doc["weightsManifest"]:
        for p in group["paths"]:
            with open(os.path.join(model_dir, p), "rb") as f:
                blobs += f.read()
        specs += group["weights"]
    arrays, off = {}, 0
    for w in specs:
        if w["dtype"] != "float32":
            raise ValueError("only float32 weights are supported")
        n = int(np.prod(w["shape"])) if w["shape"] else 1
        arrays[w["name"]] = np.frombuffer(blobs, "<f4", n, off).reshape(w["shape"]).copy()
        off += 4 * n
    kernels, biases, acts, dims = [], [], [], []
    for l in dense:
        name = l["config"]["name"]
        k = arrays[name + "/kernel"]
        b = arrays.get(name + "/bias")
        if b is None:
            b = np.zeros(k.shape[1], np.float32)
        kernels.append(np.ascontiguousarray(k, np.float32))
        biases.append(np.ascontiguousarray(b, np.float32))
        acts.append(ACTIVATIONS[l["config"]["activation"]])
        if not dims:
            dims.append(k.shape[0])
        dims.append(k.shape[1])
    nin = dims[0]
    ins = meta["inputs"]
    if meta.get("isNormalized", True):
        in_min = np.array([ins[str(i)]["min"] for i in range(nin)], np.float64)
        in_max = np.array([ins[str(i)]["max"] for i in range(nin)], np.float64)
    else:   # ml5 normalises a row only when the saved meta says the training data was (NeuralNetwork.classifyInternal)
        in_min, in_max = np.zeros(nin, np.float64), np.ones(nin, np.float64)
    labels = None
    outs = meta.get("outputs") or {}
    for o in outs.values():
        if "legend" in o:       # one-hot legend: label -> vector
            labels = [None] * len(o["legend"])
            for lab, vec in o["legend"].items():
                labels[int(np.argmax(vec))] = lab
    return dict(dims=dims, activations=acts, kernels=kernels, biases=biases, in_min=in_min, in_max=in_max,
                labels=labels or [str(i) for i in range(dims[-1])])


class Classifier:
    """A loaded model on one GPU."""

    def __init__(self, model: dict | str, device: int = 0):
        if isinstance(model, str):
            model = load_tfjs_model(model)
        self.model = model
        self.labels = list(model["labels"])
        self._lib = _capi.lib()
        n = len(model["kernels"])
        dims = (C.c_int * (n + 1))(*model["dims"])
        acts = (C.c_int * n)(*model["activations"])
        self._keep = [np.ascontiguousarray(k, np.float32) for k in model["kernels"]] + \
                     [np.ascontiguousarray(b, np.float32) for b in model["biases"]]
        kp = (C.c_void_p * n)(*[a.ctypes.data for a in self._keep[:n]])
        bp = (C.c_void_p * n)(*[a.ctypes.data for a in self._keep[n:]])
        lo = np.ascontiguousarray(model["in_min"], np.float64)
        hi = np.ascontiguousarray(model["in_max"], np.float64)
        self._h = C.c_void_p()
        rc = self._lib.fa_mlp_create(n, dims, acts, kp, bp, lo.ctypes.data, hi.ctypes.data, device, C.byref(self._h))
        if rc != 0:
            self._h = C.c_void_p()
            raise FaError(rc, self._lib.fa_status_string(rc).decode())
        self.n_in, self.n_out = model["dims"][0], model["dims"][-1]

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.fa_mlp_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def _check(self, rc):
        if rc < 0:
            raise FaError(rc, (self._lib.fa_mlp_last_error(self._h) or b"").decode() or self._lib.fa_status_string(rc).decode())
        return rc

    def probabilities(self, rows) -> np.ndarray:
        rows = np.ascontiguousarray(rows, np.float64).reshape(-1, self.n_in)
        out = np.empty((rows.shape[0], self.n_out), np.float32)
        self._check(self._lib.fa_mlp_classify(self._h, rows.ctypes.data, rows.shape[0], out.ctypes.data))
        return out

    def classify_features(self, engine, utt_id: int | None = None) -> np.ndarray:
        """Class scores of the feature rows of a finished Engine batch, computed where the rows are (device)."""
        c = engine.counts(utt_id)
        out = np.empty((c["feature_rows"], self.n_out), np.float32)
        n = self._check(self._lib.fa_mlp_classify_features(self._h, engine._h, -1 if utt_id is None else utt_id,
                                                           out.ctypes.data, out.shape[0]))
        return out[:n]

    def results(self, probs: np.ndarray) -> list:
        """ml5 classifyMultiple's shape: per row a list of {label, confidence}, highest confidence first."""
        out = []
        for p in probs:
            order = sorted(range(len(p)), key=lambda i: -float(p[i]))      # stable: ties keep label order
            out.append([{"label": self.labels[i], "confidence": float(p[i])} for i in order])
        return out

    def classify_multiple(self, rows) -> list:
        return self.results(self.probabilities(rows))


class SegmentVoter:
    """predict_by_multiple_syllables + nn_prediction + seg_confidence_sort (src/prediction.js:47-169) for one or more
    models ("DBs"): sqrt(duration)-weighted confidence sums per label, per segment and over the whole clip."""

    def __init__(self, db_ids=(1,)):
        self.db_ids = list(db_ids)
        self.conf_all = {d: {} for d in self.db_ids}
        self.sum_weights = 0.0
        self.max_inv_entropy, self.min_entropy_db = 0.0, None

    def segment(self, results_by_db: dict, seg_time) -> tuple | None:
        """results_by_db[db] = ml5-shaped results of the segment's syllable rows; seg_time = [[t0, dur] strings ...].
        Returns (top label, confidence / total duration) like the callback of predict_by_multiple_syllables."""
        seg_weight = 0.0
        for t in seg_time:          # a plain left-to-right sum like the reference's loop (Python >= 3.12's sum() compensates)
            seg_weight += float(t[1])
        if not seg_weight > 0:
            return None
        conf_seg = {d: {} for d in self.db_ids}
        for d in self.db_ids:
            res = results_by_db[d]
            for ph, t in enumerate(seg_time):
                w = math.sqrt(float(t[1]))
                # with a single syllable the app reads result_out[ph] of the FLAT class list: only the top class counts
                items = [res[0][0]] if len(seg_time) == 1 else res[ph]
                for it in items:
                    wc = it["confidence"] * w
                    self.conf_all[d][it["label"]] = self.conf_all[d].get(it["label"], 0) + wc if self.conf_all[d].get(it["label"]) else wc
                    conf_seg[d][it["label"]] = conf_seg[d].get(it["label"], 0) + wc if conf_seg[d].get(it["label"]) else wc
        self.sum_weights += seg_weight
        best, top = 0.0, None
        for d in self.db_ids:
            max_all, max_seg, lab_seg = 0.0, 0.0, None
            for lab in self.conf_all[d]:
                if self.conf_all[d][lab] > max_all:
                    max_all = self.conf_all[d][lab]
                if conf_seg[d].get(lab, 0) > max_seg:
                    max_seg, lab_seg = conf_seg[d][lab], lab
            if max_seg > best:
                best, top = max_seg, lab_seg
            if max_all > self.max_inv_entropy:
                self.max_inv_entropy, self.min_entropy_db = max_all, d
        return top, best / seg_weight


def save_tfjs_model(model: dict, model_dir: str) -> str:
    """Write `model` (the dict load_tfjs_model returns) as the files ml5 saves: model.json (tf.js layers format, weights in
    ./model.weights.bin), model.weights.bin and model_meta.json (normalised inputs with their ranges, the label legend)."""
    os.makedirs(model_dir, exist_ok=True)
    dims, labels = list(model["dims"]), list(model["labels"])
    layers, specs, blob = [], [], b""
    for i, (k, b, a) in enumerate(zip(model["kernels"], model["biases"], model["activations"])):
        name = f"dense_Dense{i + 1}"
        cfg = {"units": dims[i + 1], "activation": ACTIVATION_NAMES[int(a)], "use_bias": True, "name": name,
               "kernel_initializer": {"class_name": "GlorotUniform", "config": {"seed": None}},
               "bias_initializer": {"class_name": "Zeros", "config": {}}}
        if i == 0:
            cfg["batch_input_shape"] = [None, dims[0]]
        layers.append({"class_name": "Dense", "config": cfg})
        specs += [{"name": name + "/kernel", "shape": [dims[i], dims[i + 1]], "dtype": "float32"},
                  {"name": name + "/bias", "shape": [dims[i + 1]], "dtype": "float32"}]
        blob += np.ascontiguousarray(k, "<f4").tobytes() + np.ascontiguousarray(b, "<f4").tobytes()
    doc = {"modelTopology": {"class_name": "Sequential", "config": {"name": "sequential_1", "layers": layers},
                             "keras_version": "tfjs-layers", "backend": "tensor_flow.js"},
           "format": "layers-model", "weightsManifest": [{"paths": ["./model.weights.bin"], "weights": specs}]}
    meta = {"inputUnits": [dims[0]], "outputUnits": dims[-1],
            "inputs": {str(i): {"dtype": "number", "min": float(model["in_min"][i]), "max": float(model["in_max"][i])}
                       for i in range(dims[0])},
            "outputs": {"label": {"dtype": "string", "min": 0, "max": 1, "uniqueValues": labels,
                                  "legend": {lab: [1 if j == i else 0 for j in range(len(labels))] for i, lab in enumerate(labels)}}},
            "isNormalized": True}
    with open(os.path.join(model_dir, "model.json"), "w") as f:
        json.dump(doc, f)
    with open(os.path.join(model_dir, "model_meta.json"), "w") as f:
        json.dump(meta, f)
    with open(os.path.join(model_dir, "model.weights.bin"), "wb") as f:
        f.write(blob)
    return model_dir


def row_labels(engine, utt_labels) -> np.ndarray:
    """The app's "label from the file name" flow: utt_labels[u] (one per utterance of a finished Engine batch, in submission
    order) repeated over that utterance's feature rows, aligned with engine.feature_table()."""
    counts = engine.counts_table()["feature_rows"]
    utt_labels = np.asarray(utt_labels)
    if utt_labels.shape[0] != counts.shape[0]:
        raise ValueError(f"{utt_labels.shape[0]} labels for {counts.shape[0]} utterances")
    return np.repeat(utt_labels, counts)


def glorot_params(dims, seed: int) -> np.ndarray:
    """tf.js Dense defaults in K7's flat layout: per layer a Glorot-uniform kernel [in][out] (limit sqrt(6 / (in + out))),
    then a zero bias; drawn from numpy.random.default_rng(seed), layer after layer."""
    rng = np.random.default_rng(seed)
    parts = []
    for a, b in zip(dims[:-1], dims[1:]):
        lim = math.sqrt(6.0 / (a + b))
        parts += [rng.uniform(-lim, lim, (a, b)).astype(np.float32).ravel(), np.zeros(b, np.float32)]
    return np.concatenate(parts)


def _flat_params(model: dict) -> np.ndarray:
    parts = []
    for k, b in zip(model["kernels"], model["biases"]):
        parts += [np.asarray(k, np.float32).ravel(), np.asarray(b, np.float32).ravel()]
    return np.concatenate(parts)


def train(rows, labels, label_names, hidden=(256, 64, 16), activations="relu", optimizer: str = "adam",
          learning_rate: float | None = None, epochs: int = 32, batch_size: int = 32, seed=0, jobs=None, init: dict | None = None,
          device: int = 0):
    """Train a classifier of feature rows on the GPU (K9; one launch for all jobs and epochs).

    rows [n, d] (float64), labels [n] (int indices into label_names).  The model is d -> hidden... -> len(label_names)
    softmax, hidden layers with `activations` (one name, or one per hidden layer); with `init` (a model dict, e.g. from
    load_tfjs_model) the architecture, start weights and input ranges are init's instead (fine-tuning).  optimizer "sgd" or
    "adam"; learning_rate None takes DEFAULT_LEARNING_RATE[optimizer].  jobs None: one job on all rows, and one model is
    returned; otherwise a list of row-index arrays (repeats oversample, disjoint lists give folds) and a list of models,
    one per job.  seed: an int (job j uses seed + j: start weights and batch order) or one int per job.
    Each model is the dict load_tfjs_model returns (Classifier and save_tfjs_model take it as it is) plus
    "history": {"loss": [epochs], "accuracy": [epochs]}."""
    rows = np.ascontiguousarray(rows, np.float64)
    if rows.ndim != 2:
        raise ValueError("rows must be [n, d]")
    labels = np.ascontiguousarray(labels, np.int32).reshape(-1)
    if labels.shape[0] != rows.shape[0]:
        raise ValueError(f"{labels.shape[0]} labels for {rows.shape[0]} rows")
    label_names = [str(x) for x in label_names]
    if init is not None:
        dims, acts = [int(x) for x in init["dims"]], [int(x) for x in init["activations"]]
        if dims[0] != rows.shape[1] or dims[-1] != len(label_names):
            raise ValueError(f"init is {dims[0]} -> {dims[-1]}, the data {rows.shape[1]} -> {len(label_names)}")
    else:
        dims = [rows.shape[1], *[int(h) for h in hidden], len(label_names)]
        hid = [activations] * len(hidden) if isinstance(activations, str) else list(activations)
        if len(hid) != len(hidden):
            raise ValueError("one activation per hidden layer")
        acts = [ACTIVATIONS[a] for a in hid] + [ACTIVATIONS["softmax"]]
    if optimizer not in OPTIMIZERS:
        raise ValueError(f"optimizer must be one of {sorted(OPTIMIZERS)}")
    lr = DEFAULT_LEARNING_RATE[optimizer] if learning_rate is None else float(learning_rate)
    single = jobs is None
    job_lists = [np.arange(rows.shape[0], dtype=np.int32)] if single else [np.asarray(x, np.int32).reshape(-1) for x in jobs]
    n_jobs = len(job_lists)
    seeds = [int(seed) + j for j in range(n_jobs)] if np.isscalar(seed) else [int(s) for s in seed]
    if len(seeds) != n_jobs:
        raise ValueError(f"{len(seeds)} seeds for {n_jobs} jobs")
    offsets = np.zeros(n_jobs + 1, np.int64)
    offsets[1:] = np.cumsum([len(x) for x in job_lists])
    row_idx = np.ascontiguousarray(np.concatenate(job_lists) if n_jobs else np.zeros(0, np.int32), np.int32)
    if init is not None:
        init_params = np.tile(_flat_params(init), n_jobs)
        ranges = np.tile(np.concatenate([np.asarray(init["in_min"], np.float64), np.asarray(init["in_max"], np.float64)]), n_jobs)
    else:
        init_params = np.concatenate([glorot_params(dims, s) for s in seeds]) if n_jobs else np.zeros(0, np.float32)
        ranges = None
    n_params = sum(a * b + b for a, b in zip(dims[:-1], dims[1:]))
    nl = len(dims) - 1
    opts = _capi.FaTrainOpts(learning_rate=lr, optimizer=OPTIMIZERS[optimizer], epochs=int(epochs), batch_size=int(batch_size))
    out_params = np.empty(max(n_jobs, 1) * n_params, np.float32)
    out_ranges = np.empty((max(n_jobs, 1), 2, dims[0]), np.float64)
    history = np.empty((max(n_jobs, 1), max(int(epochs), 1), 2), np.float64)
    err = C.create_string_buffer(512)
    L = _capi.lib()
    seeds_a = np.asarray(seeds, np.uint64)
    rc = L.fa_mlp_train(nl, (C.c_int * (nl + 1))(*dims), (C.c_int * nl)(*acts), rows.ctypes.data, rows.shape[0],
                        labels.ctypes.data, n_jobs, offsets.ctypes.data, row_idx.ctypes.data, seeds_a.ctypes.data,
                        init_params.ctypes.data, None if ranges is None else ranges.ctypes.data, C.byref(opts), device,
                        out_params.ctypes.data, out_ranges.ctypes.data, history.ctypes.data, err, len(err))
    if rc != 0:
        raise FaError(rc, err.value.decode() or L.fa_status_string(rc).decode())
    models = []
    for j in range(n_jobs):
        flat, off = out_params[j * n_params: (j + 1) * n_params], 0
        kernels, biases = [], []
        for a, b in zip(dims[:-1], dims[1:]):
            kernels.append(flat[off: off + a * b].reshape(a, b).copy()); off += a * b
            biases.append(flat[off: off + b].copy()); off += b
        models.append(dict(dims=list(dims), activations=list(acts), kernels=kernels, biases=biases,
                           in_min=out_ranges[j, 0].copy(), in_max=out_ranges[j, 1].copy(), labels=list(label_names),
                           history={"loss": history[j, :epochs, 0].copy(), "accuracy": history[j, :epochs, 1].copy()}))
    return models[0] if single else models
