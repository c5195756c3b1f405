#!/usr/bin/env python
"""bench.py -- throughput of the formantanalyzer hot path on B200 (BASELINE.json metric).

A "step" is one pass of the whole hot path (K1 spectrum -> K2 peaks -> K3 segment scan -> K4 features -> K5 gather)
over one batch of synthetic speech.  Workload = BASELINE.json configs[1] (C2): 1000 utterances x 5 s x 16 kHz,
spectrum + formants output modes, producing the dB spectrum, the formant rows and the 53-dim Segment Features
(output_level 5, fftSize 2048, smoothingTimeConstant 0.8).  With --gpus N every rank runs its own 1000-utterance
batch (sharded by utterance, no data-path collective) => weak scaling.

  value     audio-seconds per second, inputs resident in HBM, CUDA events on the launching stream, max over ranks;
            --depth batches in flight (default 4: one handle + stream per slot), every step one full pass over one batch
  e2e       the same metric through the C-ABI with HOST buffers: fa_submit_pcm_batch (pinned caller PCM, zero copy),
            H2D, kernels, D2H of every result table and of the dB spectrum inside the timed region; --depth batches in
            flight, all batches drained before the clock stops
  roofline  the longest-running kernel's algorithmic bytes / its CUDA-event time vs the measured HBM peak; `kernels` has every
            kernel, `stages` the per-stage HBM and issue floors
  cpu_baseline  the CPU oracle (a restatement: kind "port") on the host cores, same workload

With --gpus N > 1 (torchrun, one rank per GPU) the workload is BASELINE.json configs[2] (C3): 48 kHz utterances, Syllable
Features (output_level 13), 12 500 utterances per GPU (100 000 on 8 GPUs), utterance u on rank u mod N, 16-bit PCM in pinned host
memory (what WAV files hold), NO data-path collective; the feature rows of all ranks are gathered on the host (gloo group) inside
the e2e timed region.  The line also carries the N-rank PCIe / host-memory floor of a step, measured in the same run with the same
buffers on all ranks at once, and the one-rank-alone figures of the same workload on the same box (weak-scaling reference).
`--workload c3` runs the same shard on one GPU.

`--impl reference` times the reference's CPU path.  The reference is browser JavaScript and this image has no JS
engine, so oracle/_ref does not exist; the arm runs the C restatement (oracle/fa_oracle.c) with OpenMP over
utterances on all host threads (kind "port").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# Hardware work queues: with the default of 8, the streams of two batches in flight (1 + sub-batches each) alias onto the
# same queue and a 1 ms segment scan falsely serialises other streams' kernels (profiles/r1_sweep_overlap.txt).
# Read by the CUDA driver at context creation, so it has to be set before torch / the library touch the device.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
# rank 0 prints ONE JSON line on stdout: keep NCCL's version banner (NCCL_DEBUG=VERSION in this image) off it
if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"

N_UTT, SECONDS, SR = 1000, 5, 16000
WORKLOAD = ("C2: 1000 synthetic 5 s 16 kHz utterances per GPU, spectrum + formants output modes + 53-dim Segment "
            "Features (output_level 5, fftSize 2048, smoothing 0.8, mel 128, step 25 ms)")
METRIC = "audio-sec/sec for 53-dim Segment Features (spectrum + formants modes)"
C3_UTT, C3_SECONDS, C3_SR, C3_HOP = 12500, 5, 48000, 1200
C3_WORKLOAD = ("C3: synthetic 5 s 48 kHz utterances, Syllable Features (output_level 13, fftSize 2048, smoothing 0.8, mel 128, "
               "step 25 ms), sharded by utterance (u mod N), int16 PCM from pinned host memory, host-side gather of the 53-dim rows")
C3_METRIC = "audio-sec/sec for 53-dim Syllable Features (sharded by utterance)"


_REAL_STDOUT = None


def capture_stdout():
    """NCCL (version banner), torchrun and friends write to fd 1: send all of that to stderr and keep the real stdout for the
    ONE JSON line the driver parses."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        os.write(1, data)
    else:
        os.write(_REAL_STDOUT, data)


def bench_config():
    from webspeechanalyzer_b200 import FaConfig
    return FaConfig.default(output_level=5, want_spectrum=1)


def make_workload(rank: int, n_utt: int):
    from webspeechanalyzer_b200 import synth_speech
    n = SECONDS * SR
    with ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:
        return list(ex.map(lambda u: synth_speech(n, SR, 20261017, rank * n_utt + u), range(n_utt)))


def bind_to_gpu_numa_node(local: int):
    """Run this rank on the CPUs of its GPU's NUMA node, so that the page-locked PCM / spectrum buffers it allocates next
    (first touch) are local to the GPU's PCIe root: the e2e path moves 1.1 GB per step per GPU over PCIe and host memory.
    Returns a short description for the JSON line; silently does nothing where sysfs does not say."""
    try:
        import torch
        props = torch.cuda.get_device_properties(local)
        bus = f"{props.pci_domain_id:04x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return {"gpu": local, "pci": bus, "numa_node": node, "cpus": len(cpus)}
    except Exception:   # noqa: BLE001  (affinity is an optimisation only)
        return None


def ncu_traffic(kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed ncu --set full capture
    (profiles/r<round>_ncu_kernels.json, written by profiles/ncu_kernels.py; the newest one); None if there is no capture."""
    import glob
    found = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_kernels.json")))     # the newest round's capture
    if not found:
        return None
    for name, d in json.load(open(found[-1])).items():   # kernel names carry template arguments ("void fa_segment_kernel<128>")
        if kernel in name:
            return d.get("dram_bytes")
    return None


def mean_candidates_per_frame(eng, utt_ids, sample: int = 16) -> float:
    """Stage 2 emits 32 bytes per candidate peak: measured on a sample of the batch (the algorithmic bytes of K2 / K3)."""
    tot, fr = 0, 0
    utt_ids = list(utt_ids)
    for i in utt_ids[:: max(1, len(utt_ids) // sample)]:
        _, cnt = eng.peak_candidates(int(i))
        tot += int(cnt.sum())
        fr += int(cnt.size)
    return tot / max(fr, 1)


def ncu_warp_instructions(kernels):
    """Warp-instructions per launch of the listed kernels (the newest profiles/r*_ncu_kernels.json), or None."""
    import glob
    found = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_kernels.json")))
    if not found:
        return None
    d = json.load(open(found[-1]))
    tot = 0.0
    for k in kernels:
        hit = [v.get("warp_instructions") for name, v in d.items() if k in name]
        if not hit or hit[0] is None:
            return None
        tot += hit[0]
    return tot


def kernel_table(stage_ms, fft_ms, alg_k, peak, with_ncu=True):
    """Per-KERNEL rows of the serial step (the spectrum stage is two launches, split by fa_spectrum_split_times; every other
    stage is one kernel): live CUDA-event ms, share of the step, algorithmic bytes of the kernel (for the two spectrum kernels
    these include the |X|/N rows the first hands the second through HBM), achieved GB/s, fraction of the measured HBM peak,
    DRAM bytes from the committed ncu capture.  Returns (rows, name of the kernel with the longest launch)."""
    ms = {"fa_fftmag_2048_kernel": float(fft_ms), "fa_smooth_bands_kernel": float(stage_ms[0] - fft_ms),
          "fa_peaks2_kernel": float(stage_ms[1]), "fa_segment2_kernel": float(stage_ms[2]), "fa_features_kernel": float(stage_ms[3])}
    rows = {}
    for k, t in ms.items():
        a = alg_k[k]
        rows[k] = {"ms": t, "share_of_step": t / max(float(stage_ms[4]), 1e-9), "algorithmic_bytes": int(a),
                   "achieved_gbs": a / (t * 1e-3) / 1e9 if t > 0 else None,
                   "frac_of_hbm_peak": a / (t * 1e-3) / 1e9 / peak if t > 0 else None,
                   "frac_of_nominal_8tbs": a / (t * 1e-3) / 1e9 / 8000.0 if t > 0 else None,
                   "ncu_dram_bytes": ncu_traffic(k) if with_ncu else None}    # the committed capture is of the C2 step
    return rows, max(ms, key=ms.get)


ISSUE_PEAK = 148 * 4 * 1.965e9     # warp-instructions per second: 148 SMs x 4 schedulers x 1 per clock at 1965 MHz


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_BYTES = 60_000_000     # --dump-outputs: array data in all (with the .npy headers, under 64 MB)


def dump_outputs(eng, out_dir: str):
    """--dump-outputs: what a caller of the timed path receives from `eng`'s last run, as out_dir/<name>.npy in float32 or
    float64 (the integer columns of the structured tables widened to float64, which holds them exactly); a table without
    rows is not written.  An array larger than its share of DUMP_BYTES is a fixed, seeded sample of its rows in row order
    (of the C2 workload: the dB spectrum), so that two builds run with the same arguments can be compared file for file."""
    eng.download()
    eng.sync()
    r = eng.result(None)

    def table(a):
        return np.stack([a[f].astype(np.float64) for f in a.dtype.names], axis=1)

    arrays = {"counts": table(eng.counts_table()), "segments": table(r.segments), "syllables": table(r.syllables),
              "formants": r.formants, "energy": r.energy, "features": r.features}
    if eng.cfg.want_spectrum:
        arrays["spectrum"] = eng.spectrum(None)
    os.makedirs(out_dir, exist_ok=True)
    cap = DUMP_BYTES // len(arrays)     # a share per output of the configuration: a sample never depends on other row counts
    for name, a in arrays.items():
        if len(a) == 0:                 # a table this output level does not fill (syllables at level 5, the C2 workload)
            continue
        a = np.ascontiguousarray(a, np.float64 if a.dtype == np.float64 else np.float32)
        if a.nbytes > cap:
            keep = np.random.default_rng(20261017).choice(len(a), cap // (a.nbytes // len(a)), replace=False)
            a = a[np.sort(keep)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def cpu_port_run(cfg, pcms, threads: int):
    """The CPU oracle over the batch, OpenMP over utterances.  Returns (seconds, frames)."""
    from oracle import oracle
    flat = np.concatenate(pcms)
    offs = np.zeros(len(pcms) + 1, np.int64)
    offs[1:] = np.cumsum([len(p) for p in pcms])
    t0 = time.perf_counter()
    frames = oracle.run_batch(cfg, flat, offs, SR, threads)
    return time.perf_counter() - t0, frames


def run_reference(args):
    """The reference's CPU implementation of the path on the host cores, on this arm's workload: C2 for one GPU, the C3
    workload when launched for several (rank 0 alone works, the others exit).  The reference is browser JavaScript and neither
    this image nor the GPU boxes carry a JS engine (probed below, reported in the line), so the arm runs the C restatement
    (oracle/fa_oracle.c, pinned against outputs of the reference's own code) with OpenMP over utterances: kind "port"."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return 0
    import shutil
    js = {name: shutil.which(name) for name in ("node", "nodejs", "deno", "bun", "qjs")}
    js_found = {k: v for k, v in js.items() if v}
    c3 = args.workload == "c3" or (args.workload == "auto" and world > 1)
    cores = os.cpu_count() or 1
    if c3:
        from oracle import oracle
        from webspeechanalyzer_b200 import synth_speech_i16_batch
        cfg = c3_config()
        n_utt = args.utts if args.utts != N_UTT else 2000       # a bounded sample of the 12 500-utterance shard
        n = C3_SECONDS * C3_SR
        i16 = synth_speech_i16_batch(np.empty(n_utt * n, np.int16), n_utt, n, C3_SR, 20261017, 0, world, threads=cores)
        flat = i16.astype(np.float32) * np.float32(1.0 / 32768.0)      # what fa_submit_pcm_i16 hands the kernels
        offs = np.arange(n_utt + 1, dtype=np.int64) * n
        sr, seconds, metric, workload = C3_SR, C3_SECONDS, C3_METRIC, C3_WORKLOAD
        sample = f"{n_utt} of {C3_UTT} utterances per GPU and step ({n_utt * seconds} s of audio), C oracle, OpenMP over utterances"

        def step(sub=None):
            m = n_utt if sub is None else sub
            t0 = time.perf_counter()
            fr = oracle.run_batch(cfg, flat[: m * n], offs[: m + 1], sr, cores)
            return time.perf_counter() - t0, fr
    else:
        cfg = bench_config()
        n_utt = args.utts
        pcms = make_workload(0, n_utt)
        sr, seconds, metric, workload = SR, SECONDS, METRIC, WORKLOAD
        sample = f"{n_utt} of {N_UTT} utterances per step ({n_utt * seconds} s of audio), C oracle, OpenMP over utterances"

        def step(sub=None):
            return cpu_port_run(cfg, pcms if sub is None else pcms[:sub], cores)
    for _ in range(args.warmup):
        step(max(8, n_utt // 10))
    t, frames = 0.0, 0
    for _ in range(args.steps):
        dt, frames = step()
        t += dt
    audio = n_utt * seconds * args.steps
    val = audio / t
    line = {"impl": "reference", "metric": metric, "value": val, "unit": "audio-s/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32 spectrum / u32 peaks / f64 features", "data": "synthetic",
            "frames_per_sec": frames * args.steps / t,
            "config": {"workload": workload, "utterances_per_step": n_utt},
            "cpu_baseline": {"value": val, "unit": "audio-s/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "js_engines_found": js_found,
            "note": "reference is browser JavaScript; no JS engine on this box (probed: node, nodejs, deno, bun, qjs), so the CPU "
                    "arm is the scalar -O2 C restatement (oracle/fa_oracle.c) with OpenMP -- a stated baseline, not the reference's "
                    "own JavaScript" if not js_found else
                    "a JS engine exists on this box: oracle/run_reference_modules.js can execute the reference's own modules here"}
    emit(line)
    return 0

def c3_config():
    from webspeechanalyzer_b200 import FaConfig
    return FaConfig.default(output_level=13, want_spectrum=0)


def run_c3(args, world, rank, local):
    """BASELINE configs[2]: the utterance-sharded Syllable-Features workload (see the module docstring)."""
    import torch
    import torch.distributed as dist

    from webspeechanalyzer_b200 import Engine, PinnedBuffer, shard, synth_speech_i16_batch
    from webspeechanalyzer_b200 import _capi
    import ctypes as C

    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local)
    host_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        host_group = dist.new_group(backend="gloo")     # the host-side gather of feature rows: no NCCL on the data path

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    cfg = c3_config()
    n_utt = args.utts if args.utts != N_UTT else C3_UTT
    n = C3_SECONDS * C3_SR
    frames_per_step = n_utt * (n // C3_HOP)
    audio_per_step = n_utt * C3_SECONDS
    # ---- the shard: utterances rank, rank + world, ... of the global set, 16-bit PCM in page-locked host memory ----
    t_gen = time.perf_counter()
    pcm = PinnedBuffer((n_utt * n,), np.int16, write_combined=bool(args.wc))
    threads = max(1, (len(os.sched_getaffinity(0)) or 1) // max(1, world))
    synth_speech_i16_batch(pcm.array, n_utt, n, C3_SR, 20261017, rank, world, threads=threads)
    offs = np.arange(n_utt + 1, dtype=np.int64) * n
    utt_ids = np.arange(n_utt, dtype=np.int64) * world + rank
    t_gen = time.perf_counter() - t_gen

    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    engs = []
    for j in range(2):
        e = Engine(cfg, device=local)
        e.set_stream(streams[j].cuda_stream)
        engs.append(e)
    eng = engs[0]

    # ---- device-resident throughput: PCM uploaded once, K passes of the whole path ----
    eng.set_pipeline(args.pipeline)
    eng.submit_batch(0, pcm.array, offs, C3_SR)
    eng.upload()
    for _ in range(max(3, args.warmup)):
        eng.run_resident()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(streams[0])
    for _ in range(args.steps):
        eng.run_resident()
    ev1.record(streams[0])
    barrier()
    ms_max = max_over_ranks(ev0.elapsed_time(ev1))
    launches_per_step = eng.launches
    if args.dump_outputs and rank == 0:
        dump_outputs(eng, args.dump_outputs)
    stage_acc = np.zeros(5)
    eng.set_pipeline(1)
    eng.run_resident()
    fft_acc = 0.0
    for _ in range(3):
        eng.run_resident()
        eng.sync()
        st = eng.stage_times()
        stage_acc += np.array([st["spectrum"], st["peaks"], st["segment"], st["features"], st["total"]])
        fft_acc += eng.spectrum_split_times()["fft"]
    stage_ms = stage_acc / 3
    fft_ms = fft_acc / 3
    eng.download()
    eng.sync()
    tot = eng.counts()
    cand_per_frame = mean_candidates_per_frame(eng, range(n_utt))     # engine-local ids (the global ones only key the gather)
    value = world * audio_per_step * args.steps / (ms_max / 1e3)

    # ---- end to end: host PCM -> device -> feature rows -> host -> gathered on rank 0 ----
    gathered = {"rows": 0, "bytes": 0}
    d2h_seen = []

    def launch(j):
        e = engs[j]
        e.reset()
        e.set_pipeline(args.e2e_pipeline)
        e.submit_batch(0, pcm.array, offs, C3_SR)      # zero copy: the H2D transfers read the pinned buffer
        e.run()                                        # asynchronous

    # the gather runs on a helper thread (gloo releases the GIL), one at a time and in step order on every rank, so that it
    # overlaps the next batch's launch and the GPU's copies instead of sitting between them; the last one is joined inside the
    # timed region.  bd: rank-local host-side breakdown of a step (seconds, summed over the timed steps)
    pool = ThreadPoolExecutor(max_workers=1)
    pending = []
    bd = {"wait_gpu": 0.0, "tables": 0.0, "gather_join": 0.0, "launch": 0.0}

    def gather_job(keys, feats):
        out = shard.gather_rows(keys, feats, dst=0, group=host_group, sort=False)
        if out is not None:
            gathered["rows"], gathered["bytes"] = int(out[1].shape[0]), int(out[0].nbytes + out[1].nbytes)

    def join_gather():
        t0 = time.perf_counter()
        while pending:
            pending.pop(0).result()
        bd["gather_join"] += time.perf_counter() - t0

    def collect(j, gather):
        e = engs[j]
        t0 = time.perf_counter()
        e.sync()
        t1 = time.perf_counter()
        ct = e.counts_table()
        feats = e.feature_table()
        d2h_seen.append(int(feats.nbytes + ct.nbytes))
        keys = shard.keys_from_counts(utt_ids, ct["feature_rows"])
        t2 = time.perf_counter()
        bd["wait_gpu"] += t1 - t0
        bd["tables"] += t2 - t1
        if gather and world > 1:      # every rank takes part (host-side gloo group); the one-rank-alone pass must not
            # at most two gathers in flight: waiting for the previous one here measured 15 ms per step at 8 ranks -- not the
            # 16 MB per rank, but the skew between ranks (a gather ends when the slowest rank has joined it)
            t3 = time.perf_counter()
            while len(pending) >= 2:
                pending.pop(0).result()
            bd["gather_join"] += time.perf_counter() - t3
            pending.append(pool.submit(gather_job, keys, feats))
        else:
            gathered["rows"], gathered["bytes"] = int(feats.shape[0]), int(keys.nbytes + feats.nbytes)

    def e2e_steps(k_steps, gather):
        inflight = []
        for k in range(k_steps):
            j = k % 2
            if len(inflight) == 2:
                collect(inflight.pop(0), gather)
            t0 = time.perf_counter()
            launch(j)
            bd["launch"] += time.perf_counter() - t0
            inflight.append(j)
        while inflight:
            collect(inflight.pop(0), gather)
        join_gather()

    e2e = None
    alone = None
    floor = None
    if not args.no_e2e:
        e2e_steps(2, True)
        barrier()
        for k in bd:
            bd[k] = 0.0
        t0 = time.perf_counter()
        e2e_steps(args.steps, True)
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        breakdown = {k: 1e3 * v / args.steps for k, v in bd.items()}
        e2e = {"value": world * audio_per_step * args.steps / dt, "unit": "audio-s/s",
               "h2d_bytes_per_step": int(pcm.array.nbytes), "d2h_bytes_per_step": int(d2h_seen[-1]),
               "ms_per_step": 1e3 * dt / args.steps, "batches_in_flight": 2,
               "gathered_rows_per_step": gathered["rows"], "gathered_bytes_per_step": gathered["bytes"],
               "rank0_host_ms_per_step": breakdown,
               "path": "per rank and step: fa_reset + fa_submit_pcm_i16_batch (pinned int16 PCM, converted on the device) + fa_run "
                       "(async) ... fa_sync + fa_copy_counts_table + fa_copy_features, then shard.gather_rows of the keyed 53-dim "
                       "rows to rank 0 over a host-side gloo group; all inside the timed region"}
        # ---- the floor of a step: the same pinned buffer copied to the device by ALL ranks at once ----
        L = _capi.lib()
        ms = C.c_float(0)

        def probe(reps):
            rc = L.fa_pcie_probe(local, C.c_void_p(pcm.array.ctypes.data), pcm.array.nbytes, reps, 0, C.byref(ms))
            if rc != 0:
                raise RuntimeError(f"fa_pcie_probe failed ({rc})")
            return float(ms.value)

        probe(1)
        barrier()
        floor_ms = max_over_ranks(probe(4))
        barrier()
        floor = {"h2d_ms_per_step_all_ranks_at_once": floor_ms, "gbps_per_gpu": pcm.array.nbytes / floor_ms / 1e6,
                 "aggregate_gbps": world * pcm.array.nbytes / floor_ms / 1e6,
                 "e2e_fraction_of_floor": floor_ms / e2e["ms_per_step"],
                 "how": "fa_pcie_probe: 4 back-to-back cudaMemcpyAsync of the step's int16 PCM from the same page-locked buffer, "
                        "CUDA events, all ranks between two barriers, max over ranks"}
        # ---- would write-combined pinned memory lift the N-rank floor?  1 GB probes of both kinds, all ranks at once
        #      (--probe-wc; measured on the 8-GPU boxes: 188 vs 190 GB/s aggregate, no) ----
        probe_bytes = 1 << 30
        kinds = {}
        for name, wc in ((("default", 0), ("write_combined", 1)) if args.probe_wc else ()):
            hb = PinnedBuffer((probe_bytes,), np.uint8, write_combined=bool(wc))
            hb.array[:: 4096] = 1                      # touch every page
            L.fa_pcie_probe(local, C.c_void_p(hb.array.ctypes.data), probe_bytes, 1, 0, C.byref(ms))
            barrier()
            rc = L.fa_pcie_probe(local, C.c_void_p(hb.array.ctypes.data), probe_bytes, 8, 0, C.byref(ms))
            t_k = max_over_ranks(float(ms.value) if rc == 0 else float("nan"))
            barrier()
            kinds[name] = {"ms_per_GiB": t_k, "gbps_per_gpu": probe_bytes / t_k / 1e6, "aggregate_gbps": world * probe_bytes / t_k / 1e6}
            hb.free()
        if kinds:
            floor["h2d_1GiB_probe_all_ranks_at_once"] = kinds
        # ---- weak-scaling reference on the same box: rank 0 alone, the other GPUs idle ----
        if world > 1:
            if rank == 0:
                e2e_steps(2, False)
                t0 = time.perf_counter()
                e2e_steps(max(3, args.steps // 2), False)
                torch.cuda.synchronize()
                dt1 = time.perf_counter() - t0
                f1 = probe(4)
                alone = {"e2e_value": audio_per_step * max(3, args.steps // 2) / dt1, "e2e_ms_per_step": 1e3 * dt1 / max(3, args.steps // 2),
                         "h2d_floor_ms": f1, "h2d_gbps": pcm.array.nbytes / f1 / 1e6}
            barrier()
    clocks = sampler.stop()
    if rank == 0:
        peak, peak_src = measured_peaks()
        N, B, hop = cfg.fft_size, cfg.bands, C3_HOP
        alg = {
            "spectrum": frames_per_step * (2 * hop + 4 * B),                                       # int16 PCM once + u32 frame (no dB rows)
            "peaks": frames_per_step * (4 * B + 32 * cand_per_frame + 12),                         # u32 frame in, 32 B per candidate + (n, g) out
            "segment": frames_per_step * (32 * cand_per_frame + 12) + tot["formant_rows"] * 48,    # candidates in, formant + energy rows out
            "features": tot["formant_rows"] * 36 + tot["feature_rows"] * 424,
        }
        names = ["spectrum", "peaks", "segment", "features"]
        shares = {k: float(stage_ms[i] / max(stage_ms[4], 1e-9)) for i, k in enumerate(names)}
        stages = {k: {"ms": float(stage_ms[i]), "share": shares[k], "algorithmic_bytes": int(alg[k]),
                      "achieved_gbs": alg[k] / (stage_ms[i] * 1e-3) / 1e9 if stage_ms[i] > 0 else None,
                      "frac_of_hbm_peak": alg[k] / (stage_ms[i] * 1e-3) / 1e9 / peak if stage_ms[i] > 0 else None}
                  for i, k in enumerate(names)}
        kernels, kern = kernel_table(stage_ms, fft_ms, {
            "fa_fftmag_2048_kernel": frames_per_step * (2 * hop + 4 * (N // 2)),      # int16 PCM once (converted on the way in), |X|/N row out
            "fa_smooth_bands_kernel": frames_per_step * (4 * (N // 2) + 4 * B),       # |X|/N row in, u32 frame out (no dB rows at this level)
            "fa_peaks2_kernel": alg["peaks"], "fa_segment2_kernel": alg["segment"], "fa_features_kernel": alg["features"]}, peak,
            with_ncu=False)
        ach = kernels[kern]["achieved_gbs"]
        line = {
            "metric": C3_METRIC, "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 spectrum / u32 peaks / f64 features", "data": "synthetic",
            "frames_per_sec": world * frames_per_step * args.steps / (ms_max / 1e3),
            "config": {"workload": C3_WORKLOAD, "utterances_per_gpu": n_utt, "utterances_total": n_utt * world,
                       "parallelism": f"shard-by-utterance x{world} (u mod N), no data-path collective, host-side gather (gloo)",
                       "pinned_pcm": "write-combined" if args.wc else "default",
                       "l2": f"inputs ({pcm.array.nbytes / 1e9:.1f} GB of PCM per step and GPU) exceed the 126 MB L2; no flush needed",
                       "workload_generation_s": t_gen},
            "roofline": {"bound": "hbm", "kernel": kern, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "traffic": None, "peak_source": peak_src, "share_of_step": kernels[kern]["share_of_step"],
                         "note": "the kernel with the longest launch of the serial step (CUDA events inside the library); the FFT "
                                 "kernel is FP32-issue bound, the segment scan / features latency bound (DESIGN.md); every kernel: "
                                 "`kernels`, by stage: `stages`"},
            "kernels": kernels, "stages": stages, "e2e": e2e, "pcie_floor": floor, "one_rank_alone_same_box": alone, "host_affinity": numa,
            "gpu_launches": int(launches_per_step * args.steps), "clocks": clocks,
            "results": {"segments": tot["segments"], "feature_rows": tot["feature_rows"], "formant_rows": tot["formant_rows"],
                        "overflow": tot["overflow"]},
        }
        emit(line)
    for e in engs:
        e.close()
    pcm.free()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--utts", type=int, default=N_UTT, help="utterances per GPU per step (default: the C2 workload)")
    ap.add_argument("--workload", default="auto", choices=["auto", "c2", "c3"],
                    help="auto: C2 on one GPU (the configuration the metric is quoted on), C3 (utterance-sharded Syllable Features) "
                         "when launched with more than one rank")
    ap.add_argument("--wc", type=int, default=0, help="C3: allocate the pinned PCM buffer write-combined (cudaHostAllocWriteCombined)")
    ap.add_argument("--probe-wc", action="store_true", help="C3: also probe the N-rank H2D floor with write-combined pinned memory")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--serial", action="store_true", help="one sub-batch (profiling: full-batch kernel launches)")
    ap.add_argument("--pipeline", type=int, default=1, help="sub-batches for the resident timed region (0 = automatic)")
    ap.add_argument("--e2e-pipeline", type=int, default=0, help="sub-batches of an e2e step (0 = automatic)")
    ap.add_argument("--depth", type=int, default=4,
                    help="batches in flight: one handle + stream per batch slot, steps alternate between them so that batch "
                         "i+1's spectrum kernels overlap batch i's (latency-bound) segment scan and PCIe copies")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0) as DIR/<name>.npy, float32 / float64, "
                         "at most 64 MB in all: a larger array is a fixed, seeded sample of its rows")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    capture_stdout()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    from webspeechanalyzer_b200 import Engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the hot path has no CPU fallback")
    if args.workload == "c3" or (args.workload == "auto" and world > 1):
        return run_c3(args, world, rank, local)
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cfg = bench_config()
    n_utt = args.utts
    pcms = make_workload(rank, n_utt)
    audio_per_step = n_utt * SECONDS
    frames_per_step = n_utt * (SECONDS * SR // 400)
    depth = 1 if args.serial else max(1, min(args.depth, 4))
    stream = torch.cuda.Stream()
    # one handle (+ its own stream and its own resident batch) per batch slot; slot j holds utterances of the same
    # synthetic family with different seeds, every step is one full pass over one 1000-utterance batch
    engs, streams = [], []
    for j in range(depth):
        e = Engine(cfg, device=local)
        sj = stream if j == 0 else torch.cuda.Stream()
        e.set_stream(sj.cuda_stream)
        e.set_pipeline(1 if args.serial else args.pipeline)
        batch = pcms if j == 0 else make_workload(rank + 1000 * j, n_utt)
        for i, p in enumerate(batch):
            e.submit(i, p, SR)
        e.upload()
        engs.append(e)
        streams.append(sj)
    eng = engs[0]

    # ---- device-resident throughput ----
    for k in range(max(3, args.warmup) * depth):
        engs[k % depth].run_resident()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stage_acc = np.zeros(5)
    barrier()
    ev0.record(stream)
    for sj in streams[1:]:
        sj.wait_event(ev0)
    for k in range(args.steps):
        engs[k % depth].run_resident()
    for sj in streams[1:]:
        stream.wait_stream(sj)
    ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches_per_step = eng.launches
    if args.dump_outputs and rank == 0:
        dump_outputs(engs[(args.steps - 1) % depth], args.dump_outputs)
    # per-stage CUDA-event times (recorded inside the library on the launching stream): a second timed region in
    # SERIAL mode (one sub-batch), because with the sub-batch pipeline the stages of different sub-batches overlap
    eng.set_pipeline(1)
    for _ in range(2):
        eng.run_resident()
    fft_acc = 0.0
    for _ in range(min(args.steps, 5)):
        eng.run_resident()
        eng.sync()
        st = eng.stage_times()
        stage_acc += np.array([st["spectrum"], st["peaks"], st["segment"], st["features"], st["total"]])
        fft_acc += eng.spectrum_split_times()["fft"]
    stage_ms = stage_acc / min(args.steps, 5)
    fft_ms = fft_acc / min(args.steps, 5)
    eng.set_pipeline(1 if args.serial else 0)
    eng.download()
    eng.sync()
    tot = eng.counts()
    cand_per_frame = mean_candidates_per_frame(eng, range(n_utt))
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * audio_per_step * args.steps / (ms_max / 1e3)

    # ---- end to end through the C-ABI with host buffers ----
    e2e = None
    edepth = min(depth, 2)      # host-buffer steps: two batches in flight keep the PCIe link busy; more only pins more memory
    if not args.no_e2e:
        M = cfg.fft_size // 2
        # the caller's buffers: page-locked host memory for the PCM batches (inputs) and for the dB spectra (outputs);
        # one set per batch slot.  A step = reset + submit one 1000-utterance batch from HOST memory + run; its results
        # (spectrum in the sink, every dense table through fa_copy_*) are read back `depth` steps later, after fa_sync,
        # so the PCIe copies of consecutive batches run back to back.  All K batches are drained inside the timed region.
        offs = np.zeros(n_utt + 1, np.int64)
        offs[1:] = np.cumsum([p.size for p in pcms])
        spec_hosts, pcm_hosts = [], []
        for j in range(edepth):
            spec_hosts.append(torch.empty((frames_per_step, M), dtype=torch.float32, pin_memory=True).numpy())
            ph = torch.empty(int(offs[-1]), dtype=torch.float32, pin_memory=True).numpy()
            for i, p in enumerate(pcms):
                ph[offs[i]: offs[i + 1]] = p
            pcm_hosts.append(ph)
        h2d = pcm_hosts[0].nbytes
        d2h_seen = []

        def launch(j):
            e = engs[j]
            e.reset()
            e.submit_batch(0, pcm_hosts[j], offs, SR)     # zero copy: H2D reads the pinned caller buffer
            e.set_spectrum_sink(spec_hosts[j])             # dB rows stream back while later sub-batches compute
            e.run()                                        # asynchronous

        def collect(j):
            e = engs[j]
            e.sync()
            r = e.result(None)
            d2h_seen.append(spec_hosts[j].nbytes + r.segments.nbytes + r.formants.nbytes + r.energy.nbytes +
                            r.features.nbytes + r.syllables.nbytes)
            return r

        def e2e_steps(k_steps):
            inflight = []
            for k in range(k_steps):
                j = k % edepth
                if len(inflight) == edepth:
                    collect(inflight.pop(0))
                launch(j)
                inflight.append(j)
            while inflight:
                collect(inflight.pop(0))

        copy_stream = torch.cuda.Stream()
        for e in engs:
            e.set_pipeline(1 if args.serial else args.e2e_pipeline)
            e.set_d2h_stream(copy_stream.cuda_stream)   # the batches' dB rows leave in submission order (FIFO on PCIe)
        e2e_steps(2 * edepth)
        barrier()
        t0 = time.perf_counter()
        e2e_steps(args.steps)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        d2h = d2h_seen[-1]
        e2e = {"value": world * audio_per_step * args.steps / float(tt.item()), "unit": "audio-s/s",
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": 1e3 * float(tt.item()) / args.steps, "batches_in_flight": edepth,
               "path": "per batch: fa_reset + fa_submit_pcm_batch (pinned host PCM) + fa_set_spectrum_sink (pinned) + fa_run "
                       "(async) ... fa_sync + fa_copy_{segments,formants,energy,syllables,features}; one handle per batch slot"}

    # ---- the same end-to-end loop for the FEATURE modes alone (Segment Features, no spectrum output), 16-bit PCM in ----
    # What a WAV-file workload looks like: int16 samples cross PCIe as they are (fa_submit_pcm_i16_batch, converted on the
    # device) and only the result tables come back.  Reported beside `e2e`; the headline `e2e` above keeps the spectrum.
    # three batches in flight here: upload, kernels and download of three different batches overlap (the float32 headline above
    # is bound by its 829 MB download alone; these modes move 160 MB in and 9 / 214 MB out, comparable to the 2 ms of kernels)
    edepth3 = max(1, min(depth, int(os.environ.get("FA_BENCH_EDEPTH", "3"))))
    e2e_feat = None
    if not args.no_e2e:
        from webspeechanalyzer_b200 import FaConfig
        cfg2 = FaConfig.default(output_level=5, want_spectrum=0)
        engs2, pcm16_hosts = [], []
        for j in range(edepth3):
            e = Engine(cfg2, device=local)
            e.set_stream(streams[j].cuda_stream)
            e.set_pipeline(1 if args.serial else args.e2e_pipeline)
            engs2.append(e)
            ph = torch.empty(int(offs[-1]), dtype=torch.int16, pin_memory=True).numpy()
            for i, p in enumerate(pcms):
                ph[offs[i]: offs[i + 1]] = np.clip(np.rint(p * 32768.0), -32768, 32767).astype(np.int16)
            pcm16_hosts.append(ph)
        seen2 = []

        def launch2(j):
            engs2[j].reset()
            engs2[j].submit_batch(0, pcm16_hosts[j], offs, SR)
            engs2[j].run()

        def collect2(j):
            engs2[j].sync()
            r = engs2[j].result(None)
            seen2.append(r.segments.nbytes + r.formants.nbytes + r.energy.nbytes + r.features.nbytes + r.syllables.nbytes)

        def steps2(k_steps):
            inflight = []
            for k in range(k_steps):
                j = k % edepth3
                if len(inflight) == edepth3:
                    collect2(inflight.pop(0))
                launch2(j)
                inflight.append(j)
            while inflight:
                collect2(inflight.pop(0))

        steps2(2 * edepth3)
        barrier()
        t0 = time.perf_counter()
        steps2(args.steps)
        torch.cuda.synchronize()
        dt2 = time.perf_counter() - t0
        tt2 = torch.tensor([dt2], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt2, op=dist.ReduceOp.MAX)
        e2e_feat = {"value": world * audio_per_step * args.steps / float(tt2.item()), "unit": "audio-s/s",
                    "h2d_bytes_per_step": int(pcm16_hosts[0].nbytes), "d2h_bytes_per_step": int(seen2[-1]),
                    "ms_per_step": 1e3 * float(tt2.item()) / args.steps, "batches_in_flight": edepth3,
                    "path": "Segment Features only (output_level 5, no spectrum output): fa_reset + fa_submit_pcm_i16_batch (pinned int16 "
                            "PCM, converted on the device) + fa_run ... fa_sync + fa_copy_{segments,formants,energy,syllables,features}"}
        for e in engs2:
            e.close()

    # ---- and with the spectrum as AnalyserNode.getByteFrequencyData (uint8 rows, a quarter of the float32 bytes), int16 PCM in ----
    e2e_byte = None
    if not args.no_e2e:
        from webspeechanalyzer_b200 import FaConfig
        M = cfg.fft_size // 2
        cfg3 = FaConfig.default(output_level=5, want_spectrum=1, spectrum_format=1)
        engs3, sinks3 = [], []
        for j in range(edepth3):
            e = Engine(cfg3, device=local)
            e.set_stream(streams[j].cuda_stream)
            e.set_pipeline(1 if args.serial else args.e2e_pipeline)
            e.set_d2h_stream(copy_stream.cuda_stream)
            engs3.append(e)
            sinks3.append(torch.empty((frames_per_step, M), dtype=torch.uint8, pin_memory=True).numpy())
        seen3 = []

        def launch3(j):
            engs3[j].reset()
            engs3[j].submit_batch(0, pcm16_hosts[j], offs, SR)
            engs3[j].set_spectrum_sink(sinks3[j])
            engs3[j].run()

        def collect3(j):
            engs3[j].sync()
            r = engs3[j].result(None)
            seen3.append(sinks3[j].nbytes + r.segments.nbytes + r.formants.nbytes + r.energy.nbytes + r.features.nbytes + r.syllables.nbytes)

        def steps3(k_steps):
            inflight = []
            for k in range(k_steps):
                j = k % edepth3
                if len(inflight) == edepth3:
                    collect3(inflight.pop(0))
                launch3(j)
                inflight.append(j)
            while inflight:
                collect3(inflight.pop(0))

        steps3(2 * edepth3)
        barrier()
        t0 = time.perf_counter()
        steps3(args.steps)
        torch.cuda.synchronize()
        dt3 = time.perf_counter() - t0
        tt3 = torch.tensor([dt3], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt3, op=dist.ReduceOp.MAX)
        e2e_byte = {"value": world * audio_per_step * args.steps / float(tt3.item()), "unit": "audio-s/s",
                    "h2d_bytes_per_step": int(pcm16_hosts[0].nbytes), "d2h_bytes_per_step": int(seen3[-1]),
                    "ms_per_step": 1e3 * float(tt3.item()) / args.steps, "batches_in_flight": edepth3,
                    "path": "the C2 outputs with the spectrum as getByteFrequencyData rows (spectrum_format FA_SPECTRUM_U8) and int16 PCM in: "
                            "fa_reset + fa_submit_pcm_i16_batch + fa_set_spectrum_sink_raw + fa_run ... fa_sync + fa_copy_*"}
        for e in engs3:
            e.close()

    clocks = sampler.stop()
    if rank == 0:
        peak, peak_src = measured_peaks()
        N, B, hop = cfg.fft_size, cfg.bands, 400
        # algorithmic bytes per unit (SURVEY.md 8(d), DESIGN.md): per frame unless noted
        alg = {
            "spectrum": frames_per_step * (4 * hop + 4 * (N // 2) + 4 * B),                       # PCM once + dB row + u32 frame
            "peaks": frames_per_step * (4 * B + 32 * cand_per_frame + 12),                         # u32 frame in, 32 B per candidate (measured count) + (n, g) out
            "segment": frames_per_step * (32 * cand_per_frame + 12) + tot["formant_rows"] * 48,    # candidates in, formant + energy rows out
            "features": tot["formant_rows"] * 36 + tot["feature_rows"] * 424,
        }
        names = ["spectrum", "peaks", "segment", "features"]
        shares = {k: float(stage_ms[i] / max(stage_ms[4], 1e-9)) for i, k in enumerate(names)}
        stage_kernels = {"spectrum": ["fa_fftmag_2048_kernel", "fa_smooth_bands_kernel"], "peaks": ["fa_peaks2_kernel"],
                         "segment": ["fa_segment2_kernel"], "features": ["fa_features_kernel"]}

        def stage_traffic(k):     # DRAM bytes per launch of the stage's kernels from the committed ncu --set full capture
            vals = [ncu_traffic(name) for name in stage_kernels[k]]
            return None if any(v is None for v in vals) else float(sum(vals))

        def issue_floor_ms(k):    # the stage's executed warp-instructions (ncu) at one per scheduler and clock
            wi = ncu_warp_instructions(stage_kernels[k])
            return None if wi is None else 1e3 * wi / ISSUE_PEAK

        stages = {k: {"ms": float(stage_ms[i]), "share": shares[k], "algorithmic_bytes": int(alg[k]),
                      "ncu_dram_bytes": stage_traffic(k),
                      "hbm_floor_ms": 1e3 * alg[k] / (peak * 1e9),
                      "issue_floor_ms": issue_floor_ms(k),
                      "frac_of_min_bound": (max(1e3 * alg[k] / (peak * 1e9), issue_floor_ms(k) or 0.0) / stage_ms[i]) if stage_ms[i] > 0 else None,
                      "achieved_gbs": alg[k] / (stage_ms[i] * 1e-3) / 1e9 if stage_ms[i] > 0 else None,
                      "frac_of_hbm_peak": alg[k] / (stage_ms[i] * 1e-3) / 1e9 / peak if stage_ms[i] > 0 else None}
                  for i, k in enumerate(names)}
        kernels, kern = kernel_table(stage_ms, fft_ms, {
            "fa_fftmag_2048_kernel": frames_per_step * (4 * hop + 4 * (N // 2)),          # PCM once, |X|/N row out
            "fa_smooth_bands_kernel": frames_per_step * (8 * (N // 2) + 4 * B),           # |X|/N row in, dB row + u32 frame out
            "fa_peaks2_kernel": alg["peaks"], "fa_segment2_kernel": alg["segment"], "fa_features_kernel": alg["features"]}, peak)
        ach = kernels[kern]["achieved_gbs"]
        line = {
            "metric": METRIC, "value": value, "unit": "audio-s/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 spectrum / u32 peaks / f64 features", "data": "synthetic",
            "frames_per_sec": world * frames_per_step * args.steps / (ms_max / 1e3),
            "config": {"workload": WORKLOAD, "utterances_per_gpu": n_utt, "parallelism": f"shard-by-utterance x{world}",
                       "batches_in_flight": depth,
                       "l2": "inputs (320 MB PCM + 819 MB spectrum rows per step) exceed the 126 MB L2; no flush needed"},
            "roofline": {"bound": "hbm", "kernel": kern, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "traffic": kernels[kern]["ncu_dram_bytes"], "peak_source": peak_src,
                         "share_of_step": kernels[kern]["share_of_step"],
                         "note": "the kernel with the longest launch of the serial step (CUDA events inside the library): the segment "
                                 "scan is a sequential state machine per utterance, latency bound -- kilobytes per utterance, so its "
                                 "fraction of the HBM peak is small by nature; the FFT kernel is FP32-issue bound, the smoothing kernel "
                                 "HBM bound.  Every kernel: `kernels`; by stage, with HBM and issue floors: `stages`; DESIGN.md section 5"},
            "kernels": kernels,
            "stages": stages,
            "e2e": e2e,
            "e2e_feature_modes": e2e_feat,
            "e2e_byte_spectrum": e2e_byte,
            "host_affinity": numa,
            "gpu_launches": int(launches_per_step * args.steps),
            "clocks": clocks,
            "results": {"segments": tot["segments"], "feature_rows": tot["feature_rows"], "formant_rows": tot["formant_rows"],
                        "overflow": tot["overflow"]},
        }
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            sub = pcms[: min(n_utt, 400)]
            cpu_port_run(cfg, sub[:16], cores)
            dt, fr = cpu_port_run(cfg, sub, cores)
            line["cpu_baseline"] = {"value": len(sub) * SECONDS / dt, "unit": "audio-s/s", "cores": cores, "kind": "port",
                                    "frames_per_sec": fr / dt,
                                    "sample": f"first {len(sub)} of {n_utt} utterances ({len(sub) * SECONDS} s of audio), C oracle, OpenMP over utterances"}
        emit(line)
    for e in engs:
        e.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
