#!/usr/bin/env python3
"""bench.py - decoded frames/s (48 kHz, 10 ms, mono, 150 B) per GPU, with HBM-roofline fraction and CPU baseline.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]
  (N > 1: launched by torchrun, one rank per GPU; streams are sharded, no collective on the data path)

A "step" is one Lc3Decoder::decode_frame (or Lc3Encoder::encode_frame) for EVERY stream of the batch: the batched hot
path, one frame per stream.  Default workload `decode48`: BASELINE.json config 5's 262,144 concurrent 48 kHz / 10 ms /
150 B mono streams, all of them on one GPU at N = 1 (they fit: 2.9 GB of codec state) and the same count on every
GPU at N > 1 (weak scaling).  Bitstreams: tests/golden/bench_c1_frames_{0,1}.npy - 1,024 distinct synthetic streams of the
SURVEY 8d corpus (200-frame clips, oracle-encoded from frame 0 by tools/make_bench_corpus.py), 8 consecutive frames
each at a per-stream offset in [10, 192], tiled over the batch.  `config.corpus` carries the statistics of what was
decoded (mean lastnz, near-empty and lsb_mode fractions), measured on the GPU from the decoder's own side information.
Other workloads (extra measurements for BASELINE.md, same JSON shape): `encode48` (config 2: 48 kHz stereo, 120 B per
channel, 4,096 stereo streams = 8,192 channels), `decode16` (config 3: 16 kHz / 7.5 ms / 30 B, 16,384 streams, LTPF
active), `roundtrip48` (config 5: encode + decode of 262,144 streams at 150 B).  Their inputs are synthetic PCM
(tools/corpus.py) and, for decode16, bitstreams produced by the GPU encoder itself.

Printed JSON (one line, rank 0):
  value        units/s with inputs resident in HBM (CUDA events on the launching stream, max over ranks, whole job)
  e2e          same metric through the host-buffer entry points: pinned host buffers in and out, every step
  roofline     dominant kernel vs the measured HBM copy bandwidth; achieved = algorithmic bytes per launch / kernel time
  cpu_baseline the oracle (C++ restatement of the reference) on the host cores, bounded sample, reported not targeted

--dump-outputs DIR writes what the last timed step returned to its caller (PCM and / or bitstreams, rank 0's streams) as
DIR/<name>.npy in float32, so that two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True          # the benchmark leaves the tree it runs from as it found it

WORKLOADS = {
    "decode48": dict(fs=48000, ms=10, nbytes=150, nf=480, streams=262144, mode="decode",
                     metric="decoded frames/sec (48kHz 10ms mono) per GPU",
                     desc="decode 48 kHz mono 10 ms, 150 B/frame, 262144 concurrent streams per GPU (BASELINE config 5's "
                          "stream count on every GPU, weak scaling), 1 frame per stream per step"),
    "encode48": dict(fs=48000, ms=10, nbytes=120, nf=480, streams=8192, mode="encode",
                     metric="encoded channel-frames/sec (48kHz 10ms, 120 B/channel) per GPU",
                     desc="encode 48 kHz stereo 10 ms at 120 B/frame/channel, 4096 stereo streams = 8192 channels per GPU "
                          "(BASELINE config 2), 1 frame per channel per step"),
    "decode16": dict(fs=16000, ms=7.5, nbytes=30, nf=120, streams=16384, mode="decode",
                     metric="decoded frames/sec (16kHz 7.5ms mono, 30 B) per GPU",
                     desc="decode 16 kHz mono 7.5 ms at 30 B/frame (LTPF and TNS active), 16384 concurrent streams per GPU "
                          "(BASELINE config 3)"),
    "mixed": dict(fs=0, ms=0, nbytes=0, nf=0, streams=65536, mode="mixed",
                  metric="decoded frames/sec (mixed 8/16/24/32/44.1/48 kHz, 7.5 and 10 ms) per GPU",
                  desc="mixed-rate batch decode: 65536 streams, stream s uses (fs_list[s mod 6], duration[(s/6) mod 2]) at "
                       "20..120 B/frame (BASELINE config 4), one Lc3MixedBatchDecoder call per step"),
    "file48": dict(fs=48000, ms=10, nbytes=150, nf=480, streams=64, frames=4096, mode="file",
                   metric="decoded frames/sec (48kHz 10ms mono, whole files, time-parallel) per GPU",
                   desc="time-parallel file decode (SURVEY 8f-1): 64 streams x 4096 consecutive frames (41 s of audio each) in "
                        "ONE lc3b_decode_stream_frames call per step, 150 B/frame"),
    "file16": dict(fs=16000, ms=7.5, nbytes=30, nf=120, streams=16384, frames=8, mode="file",
                   metric="decoded frames/sec (16kHz 7.5ms mono, 30 B, 8 frames per call, time-parallel) per GPU",
                   desc="BASELINE config 3's 16384 streams of 16 kHz / 7.5 ms / 30 B, decoded 8 consecutive frames per stream per call "
                        "with lc3b_decode_stream_frames (60 ms of audio per call): how a throughput-bound caller feeds a small "
                        "stream count"),
    "roundtrip48": dict(fs=48000, ms=10, nbytes=150, nf=480, streams=262144, mode="roundtrip",
                        metric="encode+decode round trips/sec (48kHz 10ms mono, 150 B) per GPU",
                        desc="encode then decode 48 kHz mono 10 ms at 150 B/frame, 262144 streams per GPU (BASELINE config 5)"),
}


for _k, _v in WORKLOADS.items():
    _v["name"] = _k

_JSON_FD = None


def claim_stdout():
    """Route fd 1 to stderr for the rest of the run and keep the real stdout for emit(): libraries (NCCL's version
    banner under torchrun) write to stdout, and the contract is ONE JSON line there."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, line)


NCU_RANGE = os.environ.get("LC3B_NCU_RANGE") == "1"     # ncu --profile-from-start off: capture only the first timed loop
_ncu_range_used = False


def ncu_range(start: bool):
    """cudaProfilerStart/Stop around the FIRST timed loop of the run, so that an ncu capture (tools/collect_round_profiles.sh)
    sees steady-state launches of the workload itself and none of the corpus preparation."""
    global _ncu_range_used
    if not NCU_RANGE:
        return
    import torch
    if start and not _ncu_range_used:
        torch.cuda.profiler.start()
    elif not start and not _ncu_range_used:
        torch.cuda.profiler.stop()
        _ncu_range_used = True


def algo_bytes(w):
    return w["nbytes"] + 2 * w["nf"]                  # SURVEY.md 8d: bitstream bytes + 2 bytes per PCM sample, one direction


def load_frames() -> np.ndarray:
    from tools.corpus import load_bench_c1_frames
    return load_bench_c1_frames()                                               # [1024, 8, 150] u8


DUMP_LIMIT = 60_000_000                 # bytes of float32 in all: a dump stays under 64 MB


def dump_outputs(out_dir, arrays):
    """Write each CUDA tensor of `arrays` (name -> [rows, ...]) as out_dir/<name>.npy in float32.  An array larger than
    its share of DUMP_LIMIT keeps a fixed, seeded sample of its rows, in order: the same rows on every run of a shape."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_LIMIT // len(arrays)
    for name, t in arrays.items():
        row_bytes = 4 * t[0].numel()
        if t.shape[0] * row_bytes > share:
            rows = np.sort(np.random.default_rng(0).choice(t.shape[0], max(1, share // row_bytes), replace=False))
            t = t[torch.from_numpy(rows).to(t.device)]
        np.save(Path(out_dir) / f"{name}.npy", t.float().cpu().numpy())


def gpu_corpus_stats(dev, sf, fd, frames_fsb):
    """Statistics of the bitstreams a decode workload runs on, from the GPU decoder's own inspection record
    (lc3b_decoder_set_trace): frames_fsb is a CUDA uint8 [F, U, nbytes] set of distinct streams, decoded in order."""
    import torch

    import lc3_codec_b200 as L
    F, U, nb = frames_fsb.shape
    ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(U, fd, sf, nb), dtype=torch.uint8, device=dev)
    d = L.Lc3BatchDecoder(U, fd, sf, ws, nb)
    tr, x = d.enable_trace()
    out = torch.empty((U, d.nf), dtype=torch.int16, device=dev)
    rows = []
    for f in range(F):
        d.decode_frames(16, frames_fsb[f].contiguous(), out)
        rows.append(torch.cat([tr[:, :4].clone(), tr[:, 18:19].clone(), tr[:, 21:22].clone(),
                               (x != 0).sum(1, keepdim=True).to(torch.int32)], 1))
    t = torch.stack(rows).cpu().numpy().reshape(-1, 7)
    ok = t[:, 0] == 1
    return {"distinct_streams": int(U), "frames_per_stream": int(F), "mean_lastnz": float(t[ok, 2].mean()),
            "near_empty_frac": float((t[ok, 2] <= 16).mean()), "lsb_mode_frac": float(t[ok, 3].mean()),
            "mean_nonzero_lines": float(t[ok, 6].mean()), "concealed_frac": float(1.0 - ok.mean()),
            "ltpf_active_frac": float(t[ok, 4].mean()), "tns_active_frac": float((t[ok, 5] > 0).mean()),
            "clips": "SURVEY 8d: 200 frames per stream, window of consecutive frames at a per-stream offset in [10, 192]",
            "measured": "on the GPU, lc3b_decoder_set_trace over the distinct streams before the timed region"}


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(np.max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def cpu_sample(w, cores, reps: int = 16):
    """Bounded sample of the workload for the oracle: (frames or None, pcm or None).  32 streams per host thread, each
    replaying its 8 corpus frames `reps` times, so that one call is ~0.1 s of work and thread start-up does not show."""
    from tools.corpus import make_pcm_window
    n = max(cores * 32, 64)
    if w["mode"] in ("decode", "file") and w["fs"] == 48000:
        frames = load_frames()
        frames = frames[np.arange(n) % frames.shape[0]]
        return np.ascontiguousarray(np.tile(frames, (1, reps, 1))), None
    from oracle import pyoracle as O
    lead = 4
    pcm = make_pcm_window(n, 8, w["fs"], w["nf"], lead=lead)          # same 200-frame clips and windows as the GPU arm
    frames = O.encode_streams(pcm, w["fs"], w["ms"], w["nbytes"])[:, lead:] if w["mode"] in ("decode", "file") else None
    if frames is not None:
        frames = np.ascontiguousarray(np.tile(frames, (1, reps, 1)))
    return frames, np.ascontiguousarray(np.tile(pcm[:, lead:], (1, reps, 1)))


def cpu_run(w, frames, pcm, cores):
    from oracle import pyoracle as O
    if w["mode"] in ("decode", "file"):
        O.decode_streams(frames, w["fs"], w["ms"], nthreads=cores)
        return frames.shape[0] * frames.shape[1]
    enc = O.encode_streams(pcm, w["fs"], w["ms"], w["nbytes"], nthreads=cores)
    if w["mode"] == "roundtrip":
        O.decode_streams(enc, w["fs"], w["ms"], nthreads=cores)
    return pcm.shape[0] * pcm.shape[1]


def cpu_baseline(w, target_s: float = 8.0):
    """Oracle on all host cores over a bounded sample of the same workload."""
    from oracle import pyoracle as O
    cores = O.ncores()
    frames, pcm = cpu_sample(w, cores)
    cpu_run(w, frames, pcm, cores)                                  # warm
    t0, units, reps = time.perf_counter(), 0, 0
    while time.perf_counter() - t0 < target_s:
        units += cpu_run(w, frames, pcm, cores)
        reps += 1
    dt = time.perf_counter() - t0
    shape = frames.shape if frames is not None else pcm.shape
    return {"value": units / dt, "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": f"{reps} x ({shape[0]} streams x {shape[1]} frames), {dt:.1f} s, one thread per core, "
                      "C++ restatement of lc3-codec (the Rust reference cannot be built here)"}


def cpu_baseline_mixed(target_s: float = 8.0):
    """Oracle on all host cores over the twelve configurations of the mixed-rate batch, equal stream counts each (as in
    the batch): total frames / total time."""
    from oracle import pyoracle as O
    from tools.corpus import MIXED_NBYTES, make_pcm_window
    cores = O.ncores()
    n = max(cores * 8, 64)
    samples = []
    for (fs, ms), nb in sorted(MIXED_NBYTES.items()):
        nf = O.config(fs, ms)["nf"]
        if fs == 8000:                  # no 8 kHz encoder in the reference: the committed oracle-encoded fixture
            fr = np.load(ROOT / "tests" / "golden" / f"bench_mixed_8k_{str(ms).replace('.', 'p')}ms.npy")
            fr = np.ascontiguousarray(fr[np.arange(n) % fr.shape[0]])
        else:
            fr = O.encode_streams(make_pcm_window(n, 8, fs, nf, lead=4), fs, ms, nb)[:, 4:]
        samples.append((fs, ms, np.ascontiguousarray(np.tile(fr, (1, 8, 1)))))
    for fs, ms, fr in samples:
        O.decode_streams(fr, fs, ms, nthreads=cores)                # warm
    t0, units, reps = time.perf_counter(), 0, 0
    while time.perf_counter() - t0 < target_s:
        for fs, ms, fr in samples:
            O.decode_streams(fr, fs, ms, nthreads=cores)
            units += fr.shape[0] * fr.shape[1]
        reps += 1
    dt = time.perf_counter() - t0
    return {"value": units / dt, "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": f"{reps} x (12 configurations x {n} streams x 64 frames), {dt:.1f} s, one thread per core, "
                      "C++ restatement of lc3-codec (the Rust reference cannot be built here)"}


def run_reference(args, w, rank):
    """--impl reference: the reference's CPU implementation of the path (oracle port) on the host cores."""
    if rank != 0:
        return
    from oracle import pyoracle as O
    cores = O.ncores()
    if w["mode"] == "mixed":                 # twelve configurations: the cpu_baseline leg's own loop, bounded in time
        cb = cpu_baseline_mixed(target_s=min(30.0, 0.1 * max(args.steps, 10)))
        emit(({"impl": "reference", "metric": w["metric"], "value": cb["value"], "unit": "frames/s", "n_gpus": args.gpus,
               "steps": args.steps, "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "config": {"workload": w["desc"], "note": "CPU path; bounded sample, see cpu_baseline.sample"},
               "cpu_baseline": cb,
               "e2e": {"value": cb["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    frames, pcm = cpu_sample(w, cores)
    for _ in range(args.warmup):
        cpu_run(w, frames, pcm, cores)
    t0, units = time.perf_counter(), 0
    for _ in range(args.steps):
        units += cpu_run(w, frames, pcm, cores)
    dt = time.perf_counter() - t0
    fps = units / dt
    shape = frames.shape if frames is not None else pcm.shape
    cb = {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
          "sample": f"each step processes {shape[0]} streams x {shape[1]} frames of the workload on {cores} threads"}
    emit(({
        "impl": "reference", "metric": w["metric"], "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["desc"], "note": "CPU path; a step here is a bounded sample, see cpu_baseline.sample"},
        "cpu_baseline": cb,
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank to the CPUs next to its GPU (NVML's ideal affinity) BEFORE any pinned host buffer is allocated, so
    the e2e leg's staging memory sits on the GPU's NUMA node.  One process per GPU makes this the natural placement;
    without it the ranks of a multi-GPU run share one node's memory controllers.  Best effort: silently skipped."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {64 * w_ + b for w_, word in enumerate(mask) for b in range(64) if (int(word) >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception:
        pass


def run_mixed(args, w, rank, local_rank, world, dev, dist, quick=False):
    """BASELINE config 4: twelve configurations in one batch through Lc3MixedBatchDecoder."""
    import torch

    import lc3_codec_b200 as L
    from tools.corpus import MIXED_NBYTES, make_pcm_window

    S = w["streams"]
    fs_list, dur_list = [8000, 16000, 24000, 32000, 44100, 48000], [7.5, 10]
    stream_cfg = [(fs_list[s % 6], dur_list[(s // 6) % 2]) for s in range(S)]
    dec = L.Lc3MixedBatchDecoder([(L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)) for fs, ms in stream_cfg],
                                 max_nbytes=120, device=dev)
    U, F, WARM, STRIDE = 256, 8, 4, 120
    frames = torch.zeros((F, S, STRIDE), dtype=torch.uint8, device=dev)
    lens = torch.zeros(S, dtype=torch.int32, device=dev)
    algo = 0
    for ((sf, fd), first, count), nf in zip(dec.buckets, dec.nf):
        fs = [8000, 16000, 24000, 32000, 44100, 48000][sf]
        ms = 10 if fd == 1 else 7.5
        nb = MIXED_NBYTES[(fs, ms)]
        if fs == 8000:            # committed oracle-encoded fixture (no 8 kHz encoder exists in the reference)
            fr_u = torch.from_numpy(np.load(ROOT / "tests" / "golden" / f"bench_mixed_8k_{str(ms).replace('.', 'p')}ms.npy")).to(dev)
            fr_u = fr_u.permute(1, 0, 2).contiguous()                                    # [F,U,nb]
        else:                     # bitstreams from the GPU encoder itself
            pcm_u = torch.from_numpy(make_pcm_window(U, F, fs, nf, lead=WARM)).to(dev)
            n = L.Lc3BatchEncoder.calc_working_buffer_lengths(U, L.FrameDuration(fd), L.SamplingFrequency(sf), nb)
            ews = torch.empty(n, dtype=torch.uint8, device=dev)
            enc = L.Lc3BatchEncoder(U, L.FrameDuration(fd), L.SamplingFrequency(sf), ews, nb)
            fr_all = torch.empty((WARM + F, U, nb), dtype=torch.uint8, device=dev)
            for f in range(WARM + F):
                enc.encode_frames(pcm_u[:, f].contiguous(), fr_all[f])
            torch.cuda.synchronize(dev)
            fr_u = fr_all[WARM:]
            del enc, ews
        idx = torch.arange(count, device=dev) % fr_u.shape[1]
        frames[:, first:first + count, :nb] = fr_u[:, idx]
        lens[first:first + count] = nb
        algo += count * (nb + 2 * nf)
    pcm = torch.zeros((S, 480), dtype=torch.int16, device=dev)         # a bucket writes nf of the 480: the rest stays 0
    stream = torch.cuda.current_stream(dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        barrier()
        ncu_range(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(steps):
            fn(warmup + i)
        e1.record(stream)
        barrier()
        ncu_range(False)
        ms_ = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms_], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_ = float(t.item())
        return ms_

    with ClockSampler(local_rank) as clk:
        ms_total = timed(lambda i: dec.decode_frames(16, frames[i % F], lens, pcm), args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"pcm": pcm})
    ups = world * S * args.steps / (ms_total * 1e-3)
    if quick:
        return {"quick": True, "value": ups, "unit": "frames/s", "ms_per_step": ms_total / args.steps, "streams_per_gpu": S}
    host_in = frames.cpu().pin_memory()
    host_lens = lens.cpu().pin_memory()
    host_out = [dec.alloc_host_pcm() for _ in range(2)]      # one dense pinned buffer per call in flight
    dec.set_host_pipelining(True)
    e2e_steps = max(10, min(args.steps, 100))

    def e2e_step(i):
        dec.decode_frames_host(16, host_in[i % F], host_lens, host_out[i & 1])
    for i in range(3):
        e2e_step(i)
    dec.host_fence()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(e2e_steps):
        e2e_step(3 + i)
    dec.host_fence()
    e1.record(stream)
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    if dist is not None:
        t = torch.tensor([ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = float(t.item())
    dec.set_host_pipelining(False)
    peak, peak_src = measured_peak()
    step_ms = ms_total / args.steps
    achieved = algo / (step_ms * 1e-3) / 1e9
    if rank != 0:
        return None
    cb = cpu_baseline_mixed() if (world == 1 and not args.no_cpu_baseline) else None
    return {
        "metric": w["metric"], "value": ups, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": w["desc"], "name": "mixed", "streams_per_gpu": S,
                   "parallelism": f"{world} x independent stream shards; one lc3b_mixed_decode_frames call per step = 1 entropy + "
                                  "2 dequantisation + 12 synthesis + 12 post-filter kernels as one CUDA graph"},
        "clocks": clk.summary(),
        "e2e": {"value": world * S * e2e_steps / (ms_e2e * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": S * STRIDE,
                "d2h_bytes_per_step": int(sum(c_ * n_ * 2 for (_, _, c_), n_ in zip(dec.buckets, dec.nf))),
                "ms_per_step": ms_e2e / e2e_steps,
                "api": "lc3b_mixed_decode_frames_host (Lc3MixedBatchDecoder.decode_frames_host): one H2D copy, one graph, one "
                       "dense D2H copy per step, host pipelining on, host_fence before the end event"},
        "gpu_launches": 27 * args.steps,    # entropy + 2 dequant + 12 x (synth, ltpf), issued as one graph per step
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                     "kernel": "whole step (27 kernels, one graph)", "kernel_ms": step_ms,
                     "peak_source": peak_src, "algorithmic_bytes_per_step": algo},
        "cpu_baseline": cb}


def run_file(args, w, rank, local_rank, world, dev, dist, quick=False):
    """SURVEY 8f-1: few streams, many frames - one time-parallel call per step, with the frame-by-frame path beside it."""
    import torch

    import lc3_codec_b200 as L

    S, F, NB, NF = w["streams"], w["frames"], w["nbytes"], w["nf"]
    sf, fd = L.SamplingFrequency.from_hz(w["fs"]), L.FrameDuration.from_ms(w["ms"])
    ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(S, fd, sf, NB), dtype=torch.uint8, device=dev)
    dec = L.Lc3BatchDecoder(S, fd, sf, ws, NB)
    scratch = torch.empty(dec.multi_scratch_bytes(F), dtype=torch.uint8, device=dev)
    if w["fs"] == 48000 and NB == 150:
        corpus = torch.from_numpy(load_frames()).to(dev)                              # [1024, 8, 150]
    else:                                                                             # bitstreams from the GPU encoder itself
        from tools.corpus import make_pcm_window
        U, WARM, FW = 256, 4, 8
        pcm_u = torch.from_numpy(make_pcm_window(U, FW, w["fs"], NF, lead=WARM)).to(dev)
        ews = torch.empty(L.Lc3BatchEncoder.calc_working_buffer_lengths(U, fd, sf, NB), dtype=torch.uint8, device=dev)
        enc = L.Lc3BatchEncoder(U, fd, sf, ews, NB)
        fr_all = torch.empty((WARM + FW, U, NB), dtype=torch.uint8, device=dev)
        for f in range(WARM + FW):
            enc.encode_frames(pcm_u[:, f].contiguous(), fr_all[f])
        torch.cuda.synchronize(dev)
        corpus = fr_all[WARM:].permute(1, 0, 2).contiguous()                          # [U, 8, NB]
        del enc, ews
    sidx = (torch.arange(S, device=dev) + rank * S) % corpus.shape[0]
    fidx = torch.arange(F, device=dev) % corpus.shape[1]
    frames = corpus[sidx][:, fidx].contiguous()                                       # [S, F, 150]: stream s replays its 8 frames
    pcm = torch.empty((S, F * NF), dtype=torch.int16, device=dev)
    stream = torch.cuda.current_stream(dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        barrier()
        ncu_range(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(steps):
            fn(warmup + i)
        e1.record(stream)
        barrier()
        ncu_range(False)
        ms_ = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms_], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_ = float(t.item())
        return ms_

    with ClockSampler(local_rank) as clk:
        ms_total = timed(lambda i: dec.decode_stream_frames(16, frames, pcm, scratch), args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"pcm": pcm})
    ups = world * S * F * args.steps / (ms_total * 1e-3)
    if quick:
        return {"quick": True, "value": ups, "unit": "frames/s", "ms_per_step": ms_total / args.steps, "streams_per_gpu": S,
                "frames_per_call": F}
    # the same files frame by frame (what the reference's loop shape gives a GPU): a 128-frame sample
    out1 = torch.empty((S, NF), dtype=torch.int16, device=dev)
    fb_frames = min(128, F)
    per_frame = frames.permute(1, 0, 2).contiguous()                                  # [F, S, 150]

    def fb(i):
        for f in range(fb_frames):
            dec.decode_frames(16, per_frame[f], out1)
    ms_fb = timed(fb, 2, 1)
    fb_ups = world * S * fb_frames * 2 / (ms_fb * 1e-3)
    # end to end: the files arrive in pinned host memory and the PCM goes back to pinned host memory.  The call is made on
    # CH consecutive chunks of frames (the per-stream state carries over between calls), so that the PCM copy of chunk
    # c overlaps the kernels of chunk c+1 on a second CUDA stream.
    CH = 4
    Fc = F // CH
    host_in = [frames[:, c * Fc:(c + 1) * Fc].contiguous().cpu().pin_memory() for c in range(CH)]
    host_out = [torch.empty((S, Fc * NF), dtype=torch.int16).pin_memory() for c in range(CH)]
    dev_in = [torch.empty((S, Fc, NB), dtype=torch.uint8, device=dev) for _ in range(2)]
    dev_pcm = [torch.empty((S, Fc * NF), dtype=torch.int16, device=dev) for _ in range(2)]
    scratch_c = torch.empty(dec.multi_scratch_bytes(Fc), dtype=torch.uint8, device=dev)
    copy_stream = torch.cuda.Stream(device=dev)
    copied = [None, None]

    def e2e_step(i):
        for c in range(CH):
            b = c & 1
            if copied[b] is not None:
                stream.wait_event(copied[b])                       # dev_pcm[b] has left the device
            dev_in[b].copy_(host_in[c], non_blocking=True)
            dec.decode_stream_frames(16, dev_in[b], dev_pcm[b], scratch_c)
            done = torch.cuda.Event()
            done.record(stream)
            copy_stream.wait_event(done)
            with torch.cuda.stream(copy_stream):
                host_out[c].copy_(dev_pcm[b], non_blocking=True)
                copied[b] = torch.cuda.Event()
                copied[b].record(copy_stream)

    def e2e_fence():
        for ev in copied:
            if ev is not None:
                stream.wait_event(ev)
    e2e_steps = max(5, min(args.steps, 50))
    for i in range(2):
        e2e_step(i)
    e2e_fence()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(e2e_steps):
        e2e_step(2 + i)
    e2e_fence()
    e1.record(stream)
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    if dist is not None:
        t = torch.tensor([ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = float(t.item())
    peak, peak_src = measured_peak()
    step_ms = ms_total / args.steps
    achieved = algo_bytes(w) * S * F / (step_ms * 1e-3) / 1e9
    if rank != 0:
        return None
    cb = cpu_baseline(w) if (world == 1 and not args.no_cpu_baseline) else None
    return {
        "metric": w["metric"], "value": ups, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": w["desc"], "name": w["name"], "streams_per_gpu": S, "frames_per_call": F,
                   "frame_by_frame_value": fb_ups,
                   "frame_by_frame_note": f"same handle, {fb_frames} lc3b_decode_frames calls of {S} streams each",
                   "l2": f"per-unit scratch {scratch.numel() / 1e6:.0f} MB per call, far more than the 126 MB L2",
                   "parallelism": f"{world} x independent stream shards, no collective on the data path"},
        "clocks": clk.summary(),
        "e2e": {"value": world * S * F * e2e_steps / (ms_e2e * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": S * F * NB,
                "d2h_bytes_per_step": S * F * NF * 2, "ms_per_step": ms_e2e / e2e_steps,
                "api": f"pinned host -> device copy, lc3b_decode_stream_frames (Lc3BatchDecoder.decode_stream_frames) on {CH} chunks of {Fc} "
                       "frames, device -> pinned host copy of chunk c on a second stream overlapping chunk c+1"},
        "gpu_launches": (6 + (3 * 2 if S * F >= 65536 else 0)) * args.steps,   # device-resident leg: one call (six kernels; entropy and dequantisation as four sub-batches each from 65 536 units) per step
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                     "kernel": "whole call (entropy, dequant, plc_scan, imdct_multi, ola_multi, ltpf_multi)", "kernel_ms": step_ms,
                     "peak_source": peak_src, "algorithmic_bytes_per_frame": algo_bytes(w),
                     "note": "issue/latency bound like the frame-by-frame kernels (DESIGN.md section 5)"},
        "cpu_baseline": cb,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="decode48", choices=sorted(WORKLOADS))
    ap.add_argument("--streams", type=int, default=0, help="streams per GPU (default: the named workload's)")
    ap.add_argument("--total-streams", type=int, default=0, help="strong scaling: this many streams in total, split over the GPUs")
    ap.add_argument("--distinct", type=int, default=1024, help="distinct synthetic streams the batch is tiled from (PCM workloads)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the small-batch workloads reported under `secondary`")
    ap.add_argument("--quick", action="store_true", help="device-resident loop only (for profiler captures; not a bench value)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32, a seeded row sample above 60 MB)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the GPU path: use it with --impl ours")
    claim_stdout()
    args.warmup = max(args.warmup, 3)
    w = dict(WORKLOADS[args.workload])
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    scaling = "weak"
    if args.streams:
        w["streams"] = args.streams
    if args.total_streams:
        from lc3_codec_b200.sharding import shard_range
        w["streams"] = shard_range(args.total_streams, rank, world)[1]
        scaling = "strong"
    if args.impl == "reference":
        run_reference(args, w, rank)
        return

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: lc3_codec_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    bind_to_gpu_numa_node(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    runner = {"mixed": run_mixed, "file": run_file}.get(w["mode"], run_codec)
    out = runner(args, w, rank, local_rank, world, dev, dist, quick=args.quick)
    if out is not None and not args.quick:
        out["scaling"] = scaling
        if scaling == "strong":
            out["config"]["total_streams"] = args.total_streams
        # The small-batch configurations of BASELINE.json at their stated sizes (configs 2, 3, 4), device-resident, so that
        # the driver's record of the default command carries them: latency-bound territory, see DESIGN.md section 8.
        if world == 1 and args.workload == "decode48" and not args.no_secondary:
            sec = {}
            sargs = argparse.Namespace(**vars(args))
            sargs.steps, sargs.warmup, sargs.dump_outputs = 200, 10, None
            for name in ("decode16", "mixed", "encode48", "file16"):
                ws = dict(WORKLOADS[name])
                fn = {"mixed": run_mixed, "file": run_file}.get(ws["mode"], run_codec)
                try:
                    r = fn(sargs, ws, rank, local_rank, world, dev, dist, quick=True)
                    sec[name] = {"workload": ws["desc"], "streams": ws["streams"], "ms_per_step": r["ms_per_step"],
                                 "value": r["value"], "unit": "channel-frames/s" if name == "encode48" else "frames/s"}
                    if "frames_per_call" in r:
                        sec[name]["frames_per_call"] = r["frames_per_call"]
                except Exception as e:                      # the headline must not die with a secondary measurement
                    sec[name] = {"error": repr(e)}
            out["secondary"] = sec
    if out is not None and rank == 0:
        emit(out)
    if dist is not None:
        dist.destroy_process_group()


def run_codec(args, w, rank, local_rank, world, dev, dist, quick=False):
    """decode / encode / roundtrip workloads of one (fs, duration, nbytes) configuration."""
    import torch

    import lc3_codec_b200 as L
    from tools.corpus import make_pcm_window

    S, NB, NF, mode = w["streams"], w["nbytes"], w["nf"], w["mode"]
    sf, fd = L.SamplingFrequency.from_hz(w["fs"]), L.FrameDuration.from_ms(w["ms"])
    stream = torch.cuda.current_stream(dev)
    U, F, WARM = (256 if quick and w["name"] != "decode48" else (1024 if w["name"] == "decode48" else args.distinct)), 8, 4   # distinct streams, frames each, encoder lead-in
    # rank r owns streams [r*S, (r+1)*S) of the job; stream s replays corpus stream s mod U
    idx = torch.from_numpy((np.arange(S) + rank * S) % U).to(dev)

    dec = enc = None
    ws_bytes = 0
    if mode in ("decode", "roundtrip"):
        n = L.Lc3BatchDecoder.calc_working_buffer_lengths(S, fd, sf, NB)
        ws_bytes += n
        dec_ws = torch.empty(n, dtype=torch.uint8, device=dev)
        dec = L.Lc3BatchDecoder(S, fd, sf, dec_ws, NB)
        dec.set_min_nbytes(NB)           # every frame of this workload is NB bytes: at 150 B the post filter's history is dead state
    if mode in ("encode", "roundtrip"):
        n = L.Lc3BatchEncoder.calc_working_buffer_lengths(S, fd, sf, NB)
        ws_bytes += n
        enc_ws = torch.empty(n, dtype=torch.uint8, device=dev)
        enc = L.Lc3BatchEncoder(S, fd, sf, enc_ws, NB)

    # ---- inputs, resident in HBM: [F][S][...] so that step i reads one contiguous frame set
    dev_pcm_in = dev_frames = None
    if w["name"] == "decode48":
        fr_u = torch.from_numpy(load_frames()).to(dev).permute(1, 0, 2).contiguous()                    # [F,U,150]
        dev_frames = fr_u[:, idx].contiguous()                                                           # [F,S,150]
    else:
        pcm_u = torch.from_numpy(make_pcm_window(U, F, w["fs"], NF, lead=WARM)).to(dev)                 # [U,WARM+F,nf]
        # bitstreams of the distinct streams from the GPU encoder itself (decode input / corpus statistics)
        n = L.Lc3BatchEncoder.calc_working_buffer_lengths(U, fd, sf, NB)
        tmp_ws = torch.empty(n, dtype=torch.uint8, device=dev)
        tmp_enc = L.Lc3BatchEncoder(U, fd, sf, tmp_ws, NB)
        fr_all = torch.empty((WARM + F, U, NB), dtype=torch.uint8, device=dev)
        for f in range(WARM + F):
            tmp_enc.encode_frames(pcm_u[:, f].contiguous(), fr_all[f])
        torch.cuda.synchronize(dev)
        del tmp_enc, tmp_ws
        fr_u = fr_all[WARM:].contiguous()                                                                # [F,U,NB]
        if mode == "decode":
            dev_frames = fr_u[:, idx].contiguous()                                                       # [F,S,NB]
        else:
            dev_pcm_in = pcm_u[:, WARM:][idx].permute(1, 0, 2).contiguous()                              # [F,S,nf]
    corpus_stats = gpu_corpus_stats(dev, sf, fd, fr_u) if rank == 0 else None
    del fr_u
    pcm_out = torch.empty((S, NF), dtype=torch.int16, device=dev) if dec else None
    frames_out = torch.empty((S, NB), dtype=torch.uint8, device=dev) if enc else None

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps, warmup, finish=None):
        for i in range(warmup):
            fn(i)
        if finish:
            finish()
        barrier()
        ncu_range(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(steps):
            fn(warmup + i)
        if finish:
            finish()                      # e.g. make the stream wait for the last pipelined device->host copy
        e1.record(stream)
        barrier()
        ncu_range(False)
        ms = e0.elapsed_time(e1)
        if dist is not None:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def step_dev(i):
        if mode == "decode":
            dec.decode_frames(16, dev_frames[i % F], pcm_out)
        elif mode == "encode":
            enc.encode_frames(dev_pcm_in[i % F], frames_out)
        else:
            enc.encode_frames(dev_pcm_in[i % F], frames_out)
            dec.decode_frames(16, frames_out, pcm_out)

    # decoder: entropy, dequant, synth, ltpf; encoder: mdct, ltpf, sns, tns, quantize, bs_prepare, [range_coder], bs_finish
    enc_launches = 8 if S >= 12288 else 7          # small batches run the range coder inside bs_finish (lc3b_enc_quant.cu)
    # decoder: the post-filter kernel is not launched when the min_nbytes promise rules the filter out (48 kHz: >= 110 B per
    # 10 ms); from 65 536 streams a call is issued as four sub-batches, each with its own launches (lc3b_decoder_set_split);
    # 12 288 streams and fewer take the two-kernel small-batch dequantisation
    ltpf_ruled_out = mode != "encode" and NB * 8 * (10.0 / w["ms"]) >= 560 + 80 * {8000: 0, 16000: 1, 24000: 2, 32000: 3, 44100: 4, 48000: 4}[w["fs"]]
    dec_launches = ((3 if ltpf_ruled_out else 4) + (1 if S <= 12288 else 0)) * (4 if S >= 65536 else 1)
    launches_per_step = {"decode": dec_launches, "encode": enc_launches, "roundtrip": dec_launches + enc_launches}[mode]

    # ---- device-resident throughput (value) with clocks sampled during the timed region
    with ClockSampler(local_rank) as clk:
        ms_total = timed(step_dev, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {k: v for k, v in (("frames", frames_out), ("pcm", pcm_out)) if v is not None})
    clocks = clk.summary()
    ups = world * S * args.steps / (ms_total * 1e-3)
    if quick:
        return {"quick": True, "value": ups, "unit": "frames/s", "ms_per_step": ms_total / args.steps, "streams_per_gpu": S}

    # ---- per-kernel time, each kernel alone (profiling hooks), same inputs
    k_steps = max(20, min(args.steps, 100))
    kernels_ms = {}

    def time_masks(obj, names, fn):
        for mask, name in zip((1, 2, 4), names):
            obj.set_stage_mask(mask)
            kernels_ms[name] = timed(fn, k_steps, 3) / k_steps
        obj.set_stage_mask(7)

    if enc:
        # the encoder's later kernels consume what the earlier ones leave in the workspace, so they are timed as
        # growing prefixes of the chain (masks 1, 3, 7, 15, 31, 63) and reported as differences
        prev = 0.0
        for mask, name in ((1, "lc3b::enc_mdct_kernel"), (3, "lc3b::enc_ltpf_kernel"), (7, "lc3b::enc_sns_kernel"),
                           (15, "lc3b::enc_tns_kernel"), (31, "lc3b::enc_quantize_kernel"),
                           (63, "lc3b::enc_bs_prepare+range_coder+bs_finish")):
            enc.set_stage_mask(mask)
            t = timed(lambda i: enc.encode_frames(dev_pcm_in[i % F], frames_out), k_steps, 3) / k_steps
            kernels_ms[name] = max(t - prev, 0.0)
            prev = t
        enc.set_stage_mask(63)
    if dec:
        if mode == "roundtrip":
            enc.encode_frames(dev_pcm_in[0], frames_out)           # valid bitstreams for the decoder-only timing
        time_masks(dec, ("lc3b::entropy_kernel", "lc3b::dequant_kernel", "lc3b::synth_kernel+ltpf_kernel"),
                   lambda i: dec.decode_frames(16, dev_frames[i % F] if dev_frames is not None else frames_out, pcm_out))
    dom_name = max(kernels_ms, key=kernels_ms.get)
    dom_ms = kernels_ms[dom_name]
    peak, peak_src = measured_peak()
    achieved = algo_bytes(w) * S / (dom_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "kernel": dom_name, "kernel_ms": dom_ms, "peak_source": peak_src,
                "kernels_ms": kernels_ms, "algorithmic_bytes_per_frame": algo_bytes(w),
                "note": "codec stages are issue/latency bound, not HBM bound (DESIGN.md section 5); traffic from profiles/traffic.json"}
    traffic_file = ROOT / "profiles" / "traffic.json"
    if traffic_file.exists():
        try:
            t = json.loads(traffic_file.read_text())
            per_frame = t.get("dram_bytes_per_stream_frame", {}).get(w["name"], {}).get(dom_name)
            if per_frame is not None:                  # ncu figure is per stream-frame; one launch covers S of them
                roofline["traffic"] = per_frame * S
                roofline["traffic_source"] = t.get("source")
        except Exception:
            pass

    # ---- end to end through the host-buffer entry points: pinned host in, pinned host out, every step
    e2e_steps = max(10, min(args.steps, 100))
    if mode == "decode":
        host_in = dev_frames.cpu().pin_memory()
        host_out = [torch.empty((S, NF), dtype=torch.int16).pin_memory() for _ in range(2)]
        dec.set_host_pipelining(True)       # PCM copy of step i overlaps the kernels of step i+1 (include/lc3b.h)
        ms_e2e = timed(lambda i: dec.decode_frames_host(16, host_in[i % F], host_out[i & 1]), e2e_steps, 3, finish=dec.host_fence)
        dec.set_host_pipelining(False)
        h2d, d2h = S * NB, S * NF * 2
        api = "lc3b_decode_frames_host (Lc3BatchDecoder.decode_frames_host), host pipelining on, host_fence before the end event"
    elif mode == "encode":
        host_in = dev_pcm_in.cpu().pin_memory()
        host_out = torch.empty((S, NB), dtype=torch.uint8).pin_memory()
        enc.set_host_pipelining(True)       # PCM upload of step i+1 overlaps the kernels of step i (include/lc3b.h)
        ms_e2e = timed(lambda i: enc.encode_frames_host(host_in[i % F], host_out), e2e_steps, 3)
        enc.set_host_pipelining(False)
        h2d, d2h = S * NF * 2, S * NB
        api = "lc3b_encode_frames_host (Lc3BatchEncoder.encode_frames_host), host pipelining on"
    else:
        host_in = dev_pcm_in.cpu().pin_memory()
        host_bits = torch.empty((S, NB), dtype=torch.uint8).pin_memory()
        host_out = [torch.empty((S, NF), dtype=torch.int16).pin_memory() for _ in range(2)]
        dec.set_host_pipelining(True)
        enc.set_host_pipelining(True)

        def rt(i):                          # PCM host -> bitstream host -> PCM host, as two callers of the reference would
            enc.encode_frames_host(host_in[i % F], host_bits)
            dec.decode_frames_host(16, host_bits, host_out[i & 1])
        ms_e2e = timed(rt, e2e_steps, 3, finish=dec.host_fence)
        dec.set_host_pipelining(False)
        enc.set_host_pipelining(False)
        h2d, d2h = S * (NF * 2 + NB), S * (NB + NF * 2)
        api = "lc3b_encode_frames_host then lc3b_decode_frames_host (bitstream crosses the host)"
    e2e = {"value": world * S * e2e_steps / (ms_e2e * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / e2e_steps, "api": api}

    if rank != 0:
        return None
    if True:
        cb = None
        if world == 1 and not args.no_cpu_baseline:
            cb = cpu_baseline(w)
        out = {
            "metric": w["metric"], "value": ups, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": w["desc"], "name": w["name"], "streams_per_gpu": S, "frame_bytes": NB, "nf": NF,
                       "corpus": corpus_stats,
                       "l2": f"no explicit flush: each step streams the per-stream codec state + I/O "
                             f"({ws_bytes / 1e6:.0f} MB workspace per GPU), far more than the 126 MB L2",
                       "parallelism": f"{world} x independent stream shards, no collective on the data path"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches_per_step * args.steps, "roofline": roofline,
            "cpu_baseline": cb,
        }
        return out


if __name__ == "__main__":
    main()
