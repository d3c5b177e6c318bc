"""Time-parallel encode against the frame-by-frame loop on device buffers (lc3b_encode_stream_frames).

For each shape (streams x frames) the same input is encoded twice on fresh handles: once as ONE
lc3b_encode_stream_frames call, once as F lc3b_encode_frames calls (one per frame period, device-resident views of the
same buffers, the handle's default graph mode).  Each is run once untimed (warm-up: module load, graph instantiation;
its bytes are compared) and then timed with CUDA events over a second pass of the same input, whose bytes are compared
again (both handles hold the same state by then).  48 kHz / 10 ms at 120 B per frame (BASELINE config 2's rate).

    python tools/bench_encode_stream.py [--out profiles/encode_stream_frames.json] [--shapes 2x4096,64x4096,8192x8]

Writes one JSON document with the card's name and power limit (read-only nvidia-smi query) beside the numbers.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True

FS, MS, NBYTES, NF = 48000, 10, 120, 480
PCM_PERIOD = 512        # the corpus is generated for at most 512 frames per stream and repeated along time beyond that


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clk = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def run_shape(S: int, F: int) -> dict:
    import torch

    import lc3_codec_b200 as L
    from tools.corpus import make_pcm

    sf, fd = L.SamplingFrequency.from_hz(FS), L.FrameDuration.from_ms(MS)
    base = make_pcm(S, min(F, PCM_PERIOD), FS, NF)
    pcm = np.tile(base, (1, -(-F // base.shape[1]), 1))[:, :F] if F > base.shape[1] else base
    dev = "cuda:0"
    d_pcm = torch.from_numpy(np.ascontiguousarray(pcm.reshape(S, F * NF))).to(dev)

    def encoder():
        ws = torch.empty(L.Lc3BatchEncoder.calc_working_buffer_lengths(S, fd, sf, NBYTES), dtype=torch.uint8, device=dev)
        return L.Lc3BatchEncoder(S, fd, sf, ws, NBYTES), ws

    multi, ws_m = encoder()
    single, ws_s = encoder()
    scratch = torch.empty(multi.multi_scratch_bytes(F), dtype=torch.uint8, device=dev)
    out_m = torch.zeros((S, F, NBYTES), dtype=torch.uint8, device=dev)
    out_s = torch.zeros((S, F, NBYTES), dtype=torch.uint8, device=dev)

    def one_call():
        multi.encode_stream_frames(d_pcm, out_m, scratch)

    def per_frame():
        for f in range(F):
            single.encode_frames(d_pcm[:, f * NF:(f + 1) * NF], out_s[:, f])

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    res = {"streams": S, "frames": F, "units": S * F, "scratch_bytes": int(scratch.numel()),
           "pcm": f"tools.corpus.make_pcm({S}, {min(F, PCM_PERIOD)}) repeated along time" if F > PCM_PERIOD else
                  f"tools.corpus.make_pcm({S}, {F})"}
    for p in (0, 1):                                              # pass 0: warm-up, pass 1: timed
        t_m = timed(one_call)
        t_s = timed(per_frame)
        same = bool(torch.equal(out_m, out_s))
        assert same, f"{S}x{F} pass {p}: one call and {F} frame-by-frame calls gave different bytes"
        if p == 1:
            res.update(ms_one_call=t_m, ms_frame_by_frame=t_s, speedup=t_s / t_m,
                       frames_per_s_one_call=S * F / (t_m * 1e-3), frames_per_s_frame_by_frame=S * F / (t_s * 1e-3),
                       bytes_identical=same)
    del ws_m, ws_s
    return res


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=str(ROOT / "profiles" / "encode_stream_frames.json"))
    ap.add_argument("--shapes", default="2x4096,64x4096,8192x8")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_encode_stream.py needs a CUDA device")
    doc = {"what": "lc3b_encode_stream_frames (one call) vs lc3b_encode_frames per frame period, device buffers, "
                   f"{FS} Hz / {MS} ms / {NBYTES} B", **gpu_info(), "time": time.strftime("%Y-%m-%d %H:%M:%S"),
           "shapes": []}
    for sh in args.shapes.split(","):
        S, F = (int(x) for x in sh.split("x"))
        r = run_shape(S, F)
        print(json.dumps(r), flush=True)
        doc["shapes"].append(r)
        torch.cuda.empty_cache()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(doc, indent=1) + "\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()
