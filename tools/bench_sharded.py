#!/usr/bin/env python3
"""End-to-end decode throughput through the sharded front end (lc3b_sharded_decode_frames_host, include/lc3b.h) in ONE
process: one batch in pinned host memory, one host thread + CUDA stream + device workspace per GPU, PCM back in pinned
host memory.  What a caller of the reference with host buffers and a multi-GPU box would run.

  python tools/bench_sharded.py [--gpus 1,2,4,8] [--steps 40] [--per-gpu 262144] [--total 262144]

For every GPU count G it reports
  weak    per-GPU stream count fixed (BASELINE config 5's 262,144 on every GPU), G x the work
  strong  BASELINE config 5 as written: 262,144 streams in total, split over the G GPUs
as frames/s, timed on the host around `steps` calls + wait() after 3 warm-up calls (the copies are the work here, so the
host clock is the honest one), next to the box's copy ceiling from tools/host_copy_ceiling.py when that file is present.
Bitstreams: the bench corpus (tests/golden/bench_c1_frames_{0,1}.npy), tiled.
"""
import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import lc3_codec_b200 as L  # noqa: E402
from tools.corpus import load_bench_c1_frames  # noqa: E402


def run(n_streams, devices, steps, corpus):
    F, NB, NF = corpus.shape[1], corpus.shape[2], 480
    dec = L.Lc3ShardedBatchDecoder(n_streams, L.FrameDuration.TenMs, L.SamplingFrequency.Hz48000, NB, devices=devices)
    dec.set_min_nbytes(NB)
    idx = np.arange(n_streams) % corpus.shape[0]
    host_in = torch.from_numpy(np.ascontiguousarray(corpus[idx].transpose(1, 0, 2))).pin_memory()       # [F, S, NB]
    host_out = [torch.empty((n_streams, NF), dtype=torch.int16).pin_memory() for _ in range(2)]
    for i in range(3):
        dec.decode_frames_host(16, host_in[i % F], host_out[i & 1])
    dec.wait()
    t0 = time.perf_counter()
    for i in range(steps):
        dec.decode_frames_host(16, host_in[(3 + i) % F], host_out[(3 + i) & 1])
    dec.wait()
    dt = time.perf_counter() - t0
    checksum = int(host_out[(steps + 2) & 1][:: max(1, n_streams // 64)].to(torch.int64).abs().sum())
    del dec
    return {"streams": n_streams, "gpus": len(devices), "steps": steps, "seconds": dt, "frames_per_s": n_streams * steps / dt,
            "ms_per_step": 1e3 * dt / steps, "h2d_bytes_per_step": n_streams * NB, "d2h_bytes_per_step": n_streams * NF * 2,
            "pcm_checksum": checksum}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", default="")
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--per-gpu", type=int, default=262144)
    ap.add_argument("--total", type=int, default=262144)
    a = ap.parse_args()
    have = torch.cuda.device_count()
    counts = [int(x) for x in a.gpus.split(",")] if a.gpus else [g for g in (1, 2, 4, 8) if g <= have]
    corpus = load_bench_c1_frames()
    ceiling = {}
    cf = ROOT / "profiles" / "r2_host_copy_ceiling.json"
    if cf.exists():
        for r in json.loads(cf.read_text())["rows"]:
            if r["placement"] == "default" and r["shape"] == "both":
                ceiling[r["gpus"]] = r["frames_per_s_ceiling"]
    rows = []
    for g in counts:
        devs = list(range(g))
        weak = run(a.per_gpu * g, devs, a.steps, corpus)
        strong = run(a.total, devs, a.steps, corpus)
        row = {"gpus": g, "weak": weak, "strong": strong, "copy_ceiling_frames_per_s": ceiling.get(g)}
        if ceiling.get(g):
            row["weak_fraction_of_copy_ceiling"] = weak["frames_per_s"] / ceiling[g]
        rows.append(row)
        print(json.dumps(row), flush=True)
    doc = {"what": "lc3b_sharded_decode_frames_host, one process, one host thread per GPU, pinned host buffers in and out "
                   "(tools/bench_sharded.py); decode 48 kHz / 10 ms / 150 B", "rows": rows}
    out = ROOT / "gpurun_out"
    out.mkdir(exist_ok=True)
    (out / "bench_sharded.json").write_text(json.dumps(doc, indent=1) + "\n")


if __name__ == "__main__":
    main()
