"""Subset calls (lc3b_decode_frames_subset / lc3b_encode_frames_subset) against dense handles, on device buffers.

Decoder, 48 kHz / 10 ms / 150 B (the bench fixture, tiled over the streams), a handle of 262 144 streams: for k random
distinct ids in random order, the subset call is timed against a dense handle of k streams decoding the same frames, and
at k = 262 144 also against lc3b_decode_frames on the same handle.  Encoder, 48 kHz / 10 ms / 120 B, a handle of
65 536 streams, the same comparison.  Every variant runs warm-up calls first; then the variants are timed in turns
(CUDA events around `--calls` calls, every call a new frame period, the best of `--rounds` turns), so that clock drift
hits them alike.  Also measured: the host time of a subset call (validation of the id list, the id copy, the launches;
the device drained before each call) next to a dense call's, and the graph cache statistics of a run whose k changes
every call.

    python tools/bench_subset.py [--out profiles/subset_calls.json] [--calls 20] [--rounds 3]

Writes one JSON document with the card's name and power limit (read-only nvidia-smi query) beside the numbers.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True

DEV = "cuda:0"


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clk = [x.strip() for x in q.split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def timed(fn, calls: int) -> float:
    """ms per call: CUDA events around `calls` calls of fn(i)."""
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(calls):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / calls


def race(variants: dict, calls: int, rounds: int) -> dict:
    for fn in variants.values():                                  # warm-up: module load, graphs, caches
        for i in range(3):
            fn(i)
    best = {k: float("inf") for k in variants}
    for _ in range(rounds):
        for k, fn in variants.items():
            best[k] = min(best[k], timed(fn, calls))
    return best


def host_us(fn, n: int = 20) -> float:
    """Median host time of one call with the device drained before it (microseconds)."""
    import torch
    ts = []
    for i in range(n):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn(i)
        ts.append(time.perf_counter() - t0)
    torch.cuda.synchronize()
    return float(np.median(ts) * 1e6)


def decoder_part(S: int, ks: list, calls: int, rounds: int) -> dict:
    import torch

    import lc3_codec_b200 as L
    from tools.corpus import load_bench_c1_frames

    sf, fd, NB = L.SamplingFrequency.Hz48000, L.FrameDuration.TenMs, 150
    fix = load_bench_c1_frames()                                  # [1024, 8, 150]
    P = fix.shape[1]
    d_fix = torch.from_numpy(np.ascontiguousarray(fix.transpose(1, 0, 2))).to(DEV)   # [P, 1024, 150]
    frames = [d_fix[p].repeat((S + 1023) // 1024, 1)[:S].contiguous() for p in range(P)]   # stream s: fixture row s % 1024

    def decoder(n):
        ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(n, fd, sf, NB), dtype=torch.uint8, device=DEV)
        return L.Lc3BatchDecoder(n, fd, sf, ws, NB), ws

    big, _ws = decoder(S)
    pcm = torch.empty((S, 480), dtype=torch.int16, device=DEV)
    lib = L.lib()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rng = np.random.default_rng(1)
    out = []
    for k in ks:
        ids = rng.permutation(S)[:k].astype(np.int32)
        d_ids = torch.from_numpy(ids.astype(np.int64)).to(DEV)
        sub = [frames[p].index_select(0, d_ids).contiguous() for p in range(P)]
        p_ids = C.c_void_p(ids.ctypes.data)

        def subset(i):                                            # the C entry point, without the Python wrapper
            rc = lib.lc3b_decode_frames_subset(big._h, 16, p_ids, k, C.c_void_p(sub[i % P].data_ptr()), None, NB, NB,
                                               C.c_void_p(pcm.data_ptr()), 480, None, stream)
            assert rc == 0

        dense, _wsd = decoder(k)
        pcm_d = torch.empty((k, 480), dtype=torch.int16, device=DEV)
        variants = {"subset": subset, "dense_k": lambda i: dense.decode_frames(16, sub[i % P], pcm_d)}
        if k == S:
            variants["full_call_same_handle"] = lambda i: big.decode_frames(16, frames[i % P], pcm)
        t = race(variants, calls, rounds)
        r = {"k": k, "ms_subset": t["subset"], "ms_dense_k": t["dense_k"], "subset_over_dense_k": t["subset"] / t["dense_k"]}
        if k == S:
            r.update(ms_full_call=t["full_call_same_handle"], subset_over_full_call=t["subset"] / t["full_call_same_handle"],
                     host_us_subset_call=host_us(subset),
                     host_us_full_call=host_us(lambda i: big.decode_frames(16, frames[i % P], pcm)))
            r["host_us_validation_and_id_copy"] = r["host_us_subset_call"] - r["host_us_full_call"]
        print(json.dumps(r), flush=True)
        out.append(r)
        del dense, _wsd
        torch.cuda.empty_cache()
    return {"handle_streams": S, "config": "48 kHz / 10 ms / 150 B, bench fixture tiled", "runs": out}


def encoder_part(S: int, ks: list, calls: int, rounds: int) -> dict:
    import torch

    import lc3_codec_b200 as L
    from tools.corpus import make_pcm

    sf, fd, NB, P = L.SamplingFrequency.Hz48000, L.FrameDuration.TenMs, 120, 4
    base = make_pcm(1024, P, 48000, 480)                          # stream s: the signal of stream s % 1024
    d_base = torch.from_numpy(np.ascontiguousarray(base.transpose(1, 0, 2))).to(DEV)
    pcm = [d_base[p].repeat((S + 1023) // 1024, 1)[:S].contiguous() for p in range(P)]

    def encoder(n):
        ws = torch.empty(L.Lc3BatchEncoder.calc_working_buffer_lengths(n, fd, sf, NB), dtype=torch.uint8, device=DEV)
        return L.Lc3BatchEncoder(n, fd, sf, ws, NB), ws

    big, _ws = encoder(S)
    lib = L.lib()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rng = np.random.default_rng(2)
    out = []
    for k in ks:
        ids = rng.permutation(S)[:k].astype(np.int32)
        d_ids = torch.from_numpy(ids.astype(np.int64)).to(DEV)
        sub = [pcm[p].index_select(0, d_ids).contiguous() for p in range(P)]
        y = torch.empty((k, NB), dtype=torch.uint8, device=DEV)
        p_ids = C.c_void_p(ids.ctypes.data)

        def subset(i):
            rc = lib.lc3b_encode_frames_subset(big._h, p_ids, k, C.c_void_p(sub[i % P].data_ptr()), 480,
                                               C.c_void_p(y.data_ptr()), NB, NB, stream)
            assert rc == 0

        dense, _wsd = encoder(k)
        yd = torch.empty((k, NB), dtype=torch.uint8, device=DEV)
        variants = {"subset": subset, "dense_k": lambda i: dense.encode_frames(sub[i % P], yd)}
        if k == S:
            yf = torch.empty((S, NB), dtype=torch.uint8, device=DEV)
            variants["full_call_same_handle"] = lambda i: big.encode_frames(pcm[i % P], yf)
        t = race(variants, calls, rounds)
        r = {"k": k, "ms_subset": t["subset"], "ms_dense_k": t["dense_k"], "subset_over_dense_k": t["subset"] / t["dense_k"]}
        if k == S:
            r.update(ms_full_call=t["full_call_same_handle"], subset_over_full_call=t["subset"] / t["full_call_same_handle"])
        print(json.dumps(r), flush=True)
        out.append(r)
        del dense, _wsd
        torch.cuda.empty_cache()
    return {"handle_streams": S, "config": "48 kHz / 10 ms / 120 B, tools.corpus.make_pcm(1024, 4) tiled", "runs": out}


def graph_part(S: int, calls: int) -> dict:
    """A graph-mode decoder whose call size changes every call."""
    import torch

    import lc3_codec_b200 as L
    from tools.corpus import load_bench_c1_frames

    sf, fd, NB = L.SamplingFrequency.Hz48000, L.FrameDuration.TenMs, 150
    fix = torch.from_numpy(np.ascontiguousarray(load_bench_c1_frames()[:, 0])).to(DEV)
    frames = fix.repeat((S + 1023) // 1024, 1)[:S].contiguous()
    ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(S, fd, sf, NB), dtype=torch.uint8, device=DEV)
    dec = L.Lc3BatchDecoder(S, fd, sf, ws, NB)
    dec.set_graph_mode(True)
    pcm = torch.empty((S, 480), dtype=torch.int16, device=DEV)
    rng = np.random.default_rng(3)
    sizes = rng.integers(S // 4, S + 1, calls)
    lists = [rng.permutation(S)[:n].astype(np.int32) for n in sizes]
    ms = timed(lambda i: dec.decode_frames_subset(16, lists[i], frames[:len(lists[i])], pcm[:len(lists[i])]), calls)
    return {"handle_streams": S, "calls": calls, "rows_per_call": [int(sizes.min()), int(sizes.max())],
            "ms_per_call": ms, **dec.graph_stats()}


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=str(ROOT / "profiles" / "subset_calls.json"))
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--dec-streams", type=int, default=262144)
    ap.add_argument("--dec-k", default="2048,16384,65536,262144")
    ap.add_argument("--enc-streams", type=int, default=65536)
    ap.add_argument("--enc-k", default="2048,8192,65536")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_subset.py needs a CUDA device")
    doc = {"what": "subset calls vs dense handles of the same rows and vs full calls, device buffers, CUDA events",
           **gpu_info(), "time": time.strftime("%Y-%m-%d %H:%M:%S"), "calls_per_timing": args.calls, "rounds": args.rounds}
    doc["decoder"] = decoder_part(args.dec_streams, [int(x) for x in args.dec_k.split(",")], args.calls, args.rounds)
    doc["encoder"] = encoder_part(args.enc_streams, [int(x) for x in args.enc_k.split(",")], args.calls, args.rounds)
    doc["graph_changing_k"] = graph_part(16384, 50)
    print(json.dumps(doc["graph_changing_k"]), flush=True)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(doc, indent=1) + "\n")
    print("wrote", args.out)


if __name__ == "__main__":
    main()
