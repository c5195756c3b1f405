"""K9 (csrc/fa_train.cu) on one GPU: time per epoch, steps/s, rows/s and achieved FP32 FLOP/s of classifier training, next
to the same algorithm as a plain PyTorch loop on the same GPU (baseline).

    python profiles/train_bench.py [--out FILE] [--quick]

Workloads: the shipped model 1's shape 53-256-64-16-4 on 74 249 synthetic rows (the size of its training set), batch 32,
Adam, with 1 job and with many concurrent jobs (one CTA per job); the DBs 4-7 shape 53-512-512-8 on 376 634 rows.
Per-epoch times are the difference of two runs of E1 and E2 epochs over (E2 - E1), timed with CUDA events around the call,
which ends in a device synchronise; the difference removes the upload of the rows and the range pass.  FLOPs are counted
as 6 x MAC per row (forward 2, backward 4) -- the algorithm's arithmetic, not what the kernel issues; the FP32 peak is
SMs x 128 FMA lanes x 2 x the maximum SM clock read from nvidia-smi on the box.  Card name and power limit go in the JSON."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def macs_per_row(dims):
    return sum(a * b for a, b in zip(dims[:-1], dims[1:]))


def flops_per_row_step(dims):
    return 6 * macs_per_row(dims)


def synthetic(n, n_classes, seed, d=53):
    rng = np.random.default_rng(seed)
    centres = rng.normal(0, 1, (n_classes, d))
    y = rng.integers(0, n_classes, n).astype(np.int32)
    x = (centres[y] + rng.normal(0, 1.5, (n, d))) * rng.uniform(0.5, 200, d) + rng.uniform(-50, 50, d)
    return x, y


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, check=True).stdout.splitlines()[0]
    name, power, clock = [s.strip() for s in q.split(",")]
    return name, float(power), float(clock)


def time_k9(x, y, dims, jobs, e1, e2, optimizer="adam"):
    import torch
    from webspeechanalyzer_b200 import predict
    names = [str(i) for i in range(dims[-1])]
    kw = dict(hidden=tuple(dims[1:-1]), optimizer=optimizer, batch_size=32,
              jobs=[np.arange(x.shape[0], dtype=np.int32)] * jobs, seed=list(range(jobs)))
    predict.train(x, y, names, epochs=1, **kw)                     # warm-up: module load, allocations
    ms = {}
    for e in (e1, e2):
        s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = predict.train(x, y, names, epochs=e, **kw)
        t.record()
        t.synchronize()
        ms[e] = s.elapsed_time(t)
    return (ms[e2] - ms[e1]) / (e2 - e1), out


def time_torch(x, y, dims, steps_cap=None):
    """The same algorithm in plain PyTorch (float32, min-max normalised rows, per-epoch permutation, batch 32, softmax +
    cross-entropy, Adam with tf.js constants); one epoch after a warm-up, or `steps_cap` steps scaled to an epoch."""
    import torch
    dev = torch.device("cuda")
    xt = torch.tensor(x, dtype=torch.float64, device=dev)
    lo, hi = xt.min(0).values, xt.max(0).values
    hi = torch.where(hi == lo, lo + 1, hi)
    xt = ((xt - lo) / (hi - lo)).float()
    yt = torch.tensor(y, dtype=torch.long, device=dev)
    layers = []
    for a, b in zip(dims[:-1], dims[1:]):
        layers += [torch.nn.Linear(a, b), torch.nn.ReLU()]
    net = torch.nn.Sequential(*layers[:-1]).to(dev)
    opt = torch.optim.Adam(net.parameters(), lr=1e-3, betas=(0.9, 0.999), eps=1e-7)
    n, B = x.shape[0], 32
    steps = (n + B - 1) // B if steps_cap is None else min(steps_cap, (n + B - 1) // B)

    def run(k):
        order = torch.randperm(n, device=dev)
        for s in range(k):
            idx = order[s * B: (s + 1) * B]
            loss = torch.nn.functional.cross_entropy(net(xt[idx]), yt[idx])
            opt.zero_grad(set_to_none=True)
            loss.backward()
            opt.step()

    run(50)
    torch.cuda.synchronize()
    s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    run(steps)
    t.record()
    t.synchronize()
    return s.elapsed_time(t) * ((n + B - 1) // B) / steps


def row(name, dims, n, jobs, epoch_ms, peak):
    steps = (n + 31) // 32
    fl = flops_per_row_step(dims) * n * jobs
    return {"workload": name, "dims": dims, "rows": n, "batch": 32, "jobs": jobs, "optimizer": "adam",
            "epoch_ms": round(epoch_ms, 3), "steps_per_s_per_job": round(steps / (epoch_ms / 1e3), 1),
            "rows_per_s": round(n * jobs / (epoch_ms / 1e3)), "flops_per_epoch": fl,
            "achieved_tflops": round(fl / (epoch_ms / 1e3) / 1e12, 4),
            "fraction_of_fp32_peak": round(fl / (epoch_ms / 1e3) / peak, 5)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON here (default: stdout only)")
    ap.add_argument("--quick", action="store_true", help="small sizes: a check of the script, not a measurement")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing is measured without a GPU")
    name, power, clock = card()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    peak = sms * 128 * 2 * clock * 1e6
    small, big = [53, 256, 64, 16, 4], [53, 512, 512, 8]
    n_small, n_big = (2000, 4000) if args.quick else (74249, 376634)
    res = {"card": name, "power_limit_w": power, "sm_clock_max_mhz": clock, "sms": sms,
           "fp32_fma_peak_tflops": round(peak / 1e12, 2), "flops_per_row_step": "6 x MAC (forward 2, backward 4)",
           "k9": [], "pytorch_baseline": []}
    x, y = synthetic(n_small, 4, 1)
    for jobs in (1, sms, 2 * sms):
        t0 = time.time()
        ms, _ = time_k9(x, y, small, jobs, 1, 3)
        res["k9"].append(row("53-256-64-16-4", small, n_small, jobs, ms, peak))
        print(json.dumps(res["k9"][-1]), f"({time.time() - t0:.1f} s)", flush=True)
    xb, yb = synthetic(n_big, 8, 2)
    ms, _ = time_k9(xb, yb, big, 1, 1, 2)
    res["k9"].append(row("53-512-512-8", big, n_big, 1, ms, peak))
    print(json.dumps(res["k9"][-1]), flush=True)
    for dims, (xx, yy), n in ((small, (x, y), n_small), (big, (xb, yb), n_big)):
        ms = time_torch(xx, yy, dims, steps_cap=3000)
        r = row("-".join(map(str, dims)), dims, n, 1, ms, peak)
        r["implementation"] = "PyTorch loop (torch.nn.Linear, torch.optim.Adam), 3000 steps scaled to an epoch"
        res["pytorch_baseline"].append(r)
        print(json.dumps(r), flush=True)
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
