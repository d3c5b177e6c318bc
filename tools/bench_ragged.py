"""Ragged time-parallel calls (lc3b_decode_stream_frames_subset / lc3b_encode_stream_frames_subset) against the same
schedule issued as subset calls (lc3b_decode_frames_subset / lc3b_encode_frames_subset), on device buffers.

Workloads (seeded):
  files48   1 024 streams at 48 kHz / 10 ms / 150 B (encoder: 120 B), file lengths drawn from 1 .. 1 000 frames.  One ragged
            call decodes every file; the subset schedule is one call per frame period over the files still running.
  jitter16  16 384 streams at 16 kHz / 7.5 ms / 30 B, per-period buffered depths drawn from {0, 1, 2, 3}.  One ragged call
            per period against up to three subset calls (depth 1, 2, 3) per period.
Frames are the bench fixture (48 kHz) or the engine's own encode of tools.corpus.make_pcm (16 kHz), tiled along time;
PCM input is make_pcm tiled along time.  Before timing, each pair of variants runs once on fresh handles and their
outputs are compared bit for bit.  Timing: CUDA events around the whole workload after a warm-up run, the variants in
turns, the best of --rounds.

    python tools/bench_ragged.py [--out profiles/ragged_stream_frames.json] [--rounds 3]

Writes one JSON document with the card's name and power limit (read-only nvidia-smi query) beside the numbers.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True

from tools.bench_subset import gpu_info  # noqa: E402

DEV = "cuda:0"


def timed_once(fn) -> float:
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def race(variants: dict, rounds: int) -> dict:
    for fn in variants.values():                                  # warm-up: module load, graphs, caches
        fn()
    best = {k: float("inf") for k in variants}
    for _ in range(rounds):
        for k, fn in variants.items():
            best[k] = min(best[k], timed_once(fn))
    return best


class Schedule:
    """Rows (ids, counts) of ragged calls and, for each, the subset calls of the same frames: depth d lists the rows
    with count > d, in the rows' order.  units[d]: the unit index (ragged layout) of each row of subset call d."""

    def __init__(self, ids, counts):
        self.ids, self.counts = ids.astype(np.int32), counts.astype(np.int32)
        off = np.concatenate([[0], np.cumsum(self.counts.astype(np.int64))[:-1]])
        self.total = int(self.counts.sum())
        self.sub_ids, self.units = [], []
        for d in range(int(self.counts.max(initial=0))):
            keep = self.counts > d
            self.sub_ids.append(np.ascontiguousarray(self.ids[keep]))
            self.units.append(off[keep] + d)

    def ptr(self, a):
        return C.c_void_p(a.ctypes.data)


def _p(t):
    return C.c_void_p(t.data_ptr())


def files_schedule(S, rng):
    return [Schedule(np.arange(S), rng.integers(1, 1001, S))]


def jitter_schedule(S, periods, rng):
    return [Schedule(rng.permutation(S), rng.integers(0, 4, S)) for _ in range(periods)]


def decoder_workload(name, fs, ms, nb, S, scheds, unit_frames, rounds):
    """unit_frames(sched) -> device uint8 [total, nb] (the ragged layout)."""
    import torch

    import lc3_codec_b200 as L
    sf, fd = L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)

    def decoder():
        ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(S, fd, sf, nb), dtype=torch.uint8, device=DEV)
        return L.Lc3BatchDecoder(S, fd, sf, ws, nb), ws

    frames = [unit_frames(sc) for sc in scheds]
    sub_frames = [[f.index_select(0, torch.from_numpy(u).to(DEV)).contiguous() for u in sc.units] for sc, f in zip(scheds, frames)]
    nf = L.native.config(sf, fd).nf
    pcm = [torch.empty(sc.total * nf, dtype=torch.int16, device=DEV) for sc in scheds]
    probe, _wp = decoder()
    scratch = torch.empty(max(probe.multi_subset_scratch_bytes(len(sc.ids), sc.total) for sc in scheds), dtype=torch.uint8,
                          device=DEV)
    del probe, _wp
    pcm_sub = torch.empty((S, nf), dtype=torch.int16, device=DEV)
    lib, stream = L.lib(), C.c_void_p(torch.cuda.current_stream().cuda_stream)

    # the C entry points, without the Python wrappers' argument checks
    def run_ragged(dec):
        for sc, f, p in zip(scheds, frames, pcm):
            assert lib.lc3b_decode_stream_frames_subset(dec._h, 16, sc.ptr(sc.ids), sc.ptr(sc.counts), len(sc.ids), _p(f), None,
                                                        nb, nb, _p(p), None, _p(scratch), scratch.numel(), stream) == 0

    def run_subset(dec, out=None):
        for j, (sc, sf_) in enumerate(zip(scheds, sub_frames)):
            for d, ids in enumerate(sc.sub_ids):
                assert lib.lc3b_decode_frames_subset(dec._h, 16, sc.ptr(ids), len(ids), _p(sf_[d]), None, nb, nb, _p(pcm_sub), nf,
                                                     None, stream) == 0
                if out is not None:
                    out[j].view(-1, nf).index_copy_(0, torch.from_numpy(sc.units[d]).to(DEV), pcm_sub[:len(ids)])

    a, _wa = decoder()
    run_ragged(a)
    b, _wb = decoder()
    check = [torch.empty_like(p) for p in pcm]
    run_subset(b, check)
    torch.cuda.synchronize()
    identical = all(torch.equal(p, q) for p, q in zip(pcm, check))
    assert identical, f"{name}: ragged and subset PCM differ"
    t = race({"ragged": lambda: run_ragged(a), "subset": lambda: run_subset(b)}, rounds)
    return _result(name, fs, ms, nb, S, scheds, t, identical)


def encoder_workload(name, fs, ms, nb, S, scheds, unit_pcm, rounds):
    """unit_pcm(sched) -> device int16 [total, nf] (the ragged layout)."""
    import torch

    import lc3_codec_b200 as L
    sf, fd = L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)

    def encoder():
        ws = torch.empty(L.Lc3BatchEncoder.calc_working_buffer_lengths(S, fd, sf, nb), dtype=torch.uint8, device=DEV)
        return L.Lc3BatchEncoder(S, fd, sf, ws, nb), ws

    pcm = [unit_pcm(sc) for sc in scheds]
    sub_pcm = [[x.index_select(0, torch.from_numpy(u).to(DEV)).contiguous() for u in sc.units] for sc, x in zip(scheds, pcm)]
    out = [torch.empty((sc.total, nb), dtype=torch.uint8, device=DEV) for sc in scheds]
    probe, _wp = encoder()
    scratch = torch.empty(max(probe.multi_subset_scratch_bytes(len(sc.ids), sc.total) for sc in scheds), dtype=torch.uint8,
                          device=DEV)
    del probe, _wp
    out_sub = torch.empty((S, nb), dtype=torch.uint8, device=DEV)
    nf = pcm[0].shape[1]
    lib, stream = L.lib(), C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def run_ragged(enc):
        for sc, x, y in zip(scheds, pcm, out):
            assert lib.lc3b_encode_stream_frames_subset(enc._h, sc.ptr(sc.ids), sc.ptr(sc.counts), len(sc.ids), _p(x), _p(y), nb,
                                                        nb, _p(scratch), scratch.numel(), stream) == 0

    def run_subset(enc, res=None):
        for j, (sc, xs) in enumerate(zip(scheds, sub_pcm)):
            for d, ids in enumerate(sc.sub_ids):
                assert lib.lc3b_encode_frames_subset(enc._h, sc.ptr(ids), len(ids), _p(xs[d]), nf, _p(out_sub), nb, nb,
                                                     stream) == 0
                if res is not None:
                    res[j].index_copy_(0, torch.from_numpy(sc.units[d]).to(DEV), out_sub[:len(ids)])

    a, _wa = encoder()
    run_ragged(a)
    b, _wb = encoder()
    check = [torch.empty_like(y) for y in out]
    run_subset(b, check)
    torch.cuda.synchronize()
    identical = all(torch.equal(y, z) for y, z in zip(out, check))
    assert identical, f"{name}: ragged and subset bytes differ"
    t = race({"ragged": lambda: run_ragged(a), "subset": lambda: run_subset(b)}, rounds)
    return _result(name, fs, ms, nb, S, scheds, t, identical)


def _result(name, fs, ms, nb, S, scheds, t, identical):
    frames = sum(sc.total for sc in scheds)
    r = {"workload": name, "config": f"{fs // 1000} kHz / {ms} ms / {nb} B", "streams": S, "ragged_calls": len(scheds),
         "subset_calls": sum(len(sc.sub_ids) for sc in scheds), "frames": frames,
         "ms_ragged": t["ragged"], "ms_subset": t["subset"],
         "M_frames_per_s_ragged": frames / t["ragged"] / 1e3, "M_frames_per_s_subset": frames / t["subset"] / 1e3,
         "subset_over_ragged": t["subset"] / t["ragged"], "outputs_bit_identical": identical}
    print(json.dumps(r), flush=True)
    return r


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=str(ROOT / "profiles" / "ragged_stream_frames.json"))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--jitter-periods", type=int, default=20)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_ragged.py needs a CUDA device")

    import lc3_codec_b200 as L
    from tools.corpus import load_bench_c1_frames, make_pcm

    rng = np.random.default_rng(7)
    files = files_schedule(1024, rng)
    jitter = jitter_schedule(16384, args.jitter_periods, rng)

    def tiled_units(base, sc):
        """base [B, P, ...] on the device; unit f of row i = base[ids[i] % B, f % P]."""
        B, P = base.shape[0], base.shape[1]
        s = np.repeat(sc.ids, sc.counts) % B
        f = np.concatenate([np.arange(c) for c in sc.counts]) % P if sc.total else np.zeros(0, np.int64)
        return base[torch.from_numpy(s.astype(np.int64)).to(DEV), torch.from_numpy(f.astype(np.int64)).to(DEV)].contiguous()

    fix48 = torch.from_numpy(load_bench_c1_frames()).to(DEV)                       # [1024, 8, 150]
    pcm48 = torch.from_numpy(make_pcm(1024, 8, 48000, 480)).to(DEV)
    pcm16 = make_pcm(1024, 8, 16000, 120)
    ws = torch.empty(L.Lc3BatchEncoder.calc_working_buffer_lengths(1024, L.FrameDuration.SevenPointFiveMs,
                                                                   L.SamplingFrequency.Hz16000, 30), dtype=torch.uint8, device=DEV)
    enc16 = L.Lc3BatchEncoder(1024, L.FrameDuration.SevenPointFiveMs, L.SamplingFrequency.Hz16000, ws, 30)
    fr16 = torch.empty((1024, 8, 30), dtype=torch.uint8, device=DEV)
    enc16.encode_stream_frames(torch.from_numpy(pcm16.reshape(1024, -1)).to(DEV), fr16,
                               torch.empty(enc16.multi_scratch_bytes(8), dtype=torch.uint8, device=DEV))
    pcm16 = torch.from_numpy(pcm16).to(DEV)
    del enc16, ws

    doc = {"what": "one ragged time-parallel call vs the same schedule as subset calls, device buffers, CUDA events around "
                   "the whole workload, best of rounds", **gpu_info(), "time": time.strftime("%Y-%m-%d %H:%M:%S"),
           "rounds": args.rounds, "runs": []}
    runs = doc["runs"]
    runs.append(decoder_workload("decode files48", 48000, 10, 150, 1024, files, lambda sc: tiled_units(fix48, sc), args.rounds))
    runs.append(decoder_workload("decode jitter16", 16000, 7.5, 30, 16384, jitter, lambda sc: tiled_units(fr16, sc), args.rounds))
    torch.cuda.empty_cache()
    runs.append(encoder_workload("encode files48", 48000, 10, 120, 1024, files, lambda sc: tiled_units(pcm48, sc), args.rounds))
    runs.append(encoder_workload("encode jitter16", 16000, 7.5, 30, 16384, jitter, lambda sc: tiled_units(pcm16, sc), args.rounds))
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(doc, indent=1) + "\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()
