#!/usr/bin/env python3
"""Loss / corruption harness (SURVEY.md 8f-3): fault injection over a batch of streams and a batched comparison of the
engine's concealment and recovery with the oracle's.

The reference conceals every bitstream error and returns Ok (src/decoder/lc3_decoder.rs:138-141,
src/decoder/packet_loss_concealment.rs:63-85); the error detail it computes (arithmetic_codec.rs:28-49,
side_info_reader.rs:14-21) is discarded.  The engine keeps that contract: `status_out` says concealed or not, nothing
more - a decoder that told the caller more than the reference does would not be a drop-in, and the concealment output
does not depend on which error it was.

Fault models (deterministic per seed):
  drop      Gilbert-Elliott frame loss: good->bad with p_gb, bad->good with p_bg (mean burst 1/p_bg frames); len = 0
  flip      every frame is hit with probability p_flip by 1..4 single-bit flips
  truncate  with probability p_trunc the frame is delivered short (only its first len' bytes, len' uniform in [2, nbytes))
  garbage   with probability p_garbage the whole frame is replaced by random bytes

`run()` decodes the damaged batch with the oracle and with the engine (frame by frame and, optionally, through the
time-parallel entry point) and reports: concealed-flag agreement, PCM agreement, and the recovery distance (frames after
the end of a concealed run until the damaged decode is back within +-1 LSB of the clean decode).

  python tools/loss_harness.py --fs 48000 --ms 10 --nbytes 150 --streams 2048 --frames 64      (needs a GPU)
"""
from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))


def inject(frames: np.ndarray, seed: int = 1, p_gb: float = 0.03, p_bg: float = 0.4, p_flip: float = 0.05,
           p_trunc: float = 0.01, p_garbage: float = 0.01):
    """frames [S,F,nbytes] u8 -> (damaged frames, lens [S,F] i32, kind [S,F] u8: 0 clean 1 drop 2 flip 3 truncate 4 garbage)."""
    rng = np.random.default_rng(seed)
    S, F, nb = frames.shape
    out = frames.copy()
    lens = np.full((S, F), nb, np.int32)
    kind = np.zeros((S, F), np.uint8)
    # Gilbert-Elliott loss, vectorised over streams
    bad = np.zeros(S, bool)
    u = rng.random((S, F))
    for f in range(F):
        bad = np.where(bad, u[:, f] >= p_bg, u[:, f] < p_gb)
        kind[bad, f] = 1
    lens[kind == 1] = 0
    r = rng.random((S, F))
    clean = kind == 0
    sel = clean & (r < p_flip)
    for s, f in np.argwhere(sel):
        for _ in range(int(rng.integers(1, 5))):
            out[s, f, rng.integers(0, nb)] ^= np.uint8(1 << int(rng.integers(0, 8)))
    kind[sel] = 2
    sel = clean & (r >= p_flip) & (r < p_flip + p_trunc)
    for s, f in np.argwhere(sel):
        lens[s, f] = int(rng.integers(2, nb))
    kind[sel] = 3
    sel = clean & (r >= p_flip + p_trunc) & (r < p_flip + p_trunc + p_garbage)
    n = int(sel.sum())
    if n:
        out[sel] = rng.integers(0, 256, size=(n, nb), dtype=np.uint8)
    kind[sel] = 4
    return out, lens, kind


def recovery_distance(clean_pcm: np.ndarray, damaged_pcm: np.ndarray, concealed: np.ndarray, horizon: int = 8):
    """For every end of a concealed run: frames until |damaged - clean| <= 1 LSB on a whole frame (horizon if never)."""
    S, F, _ = clean_pcm.shape
    close = (np.abs(clean_pcm.astype(np.int32) - damaged_pcm.astype(np.int32)).max(-1) <= 1)
    ends = concealed[:, :-1] & ~concealed[:, 1:]
    dist = []
    for s, f in np.argwhere(ends):
        d = horizon
        for j in range(1, horizon + 1):
            g = f + j
            if g >= F or concealed[s, g]:
                d = None                      # the next damage arrives first: not a measurement
                break
            if close[s, g]:
                d = j
                break
        if d is not None:
            dist.append(d)
    return np.asarray(dist, np.int32)


def run(fs: int, ms: float, nbytes: int, n_streams: int, n_frames: int, seed: int = 1, multi: bool = True, **fault):
    """Returns a report dict; raises AssertionError where the engine and the oracle disagree."""
    import torch

    import lc3_codec_b200 as L
    from common import corpus, gpu_decode
    from oracle import pyoracle as O

    _, frames = corpus(fs, ms, nbytes, n_streams, n_frames)
    damaged, lens, kind = inject(frames, seed, **fault)
    o_pcm, o_tr, _, _ = O.decode_streams(damaged, fs, ms, lens, trace=True)
    o_clean = O.decode_streams(frames, fs, ms)
    g_pcm, g_tr, _, _, g_status = gpu_decode(fs, ms, damaged, lens)
    o_concealed = o_tr[..., 0] == 0
    assert np.array_equal(g_status != 0, o_concealed), "concealed flags differ from the oracle's"
    assert np.array_equal(o_tr, g_tr), "decoded side information differs on the frames that survived"
    e_pcm = O.decode_streams(damaged, fs, ms, lens, transform="engine")
    assert np.array_equal(g_pcm, e_pcm), "PCM not bit exact against the oracle with the engine's inverse MDCT"
    diff = np.abs(o_pcm.astype(np.int32) - g_pcm.astype(np.int32))
    assert diff.max() <= 1, f"PCM differs by {diff.max()} LSB"
    rep = {
        "config": {"fs": fs, "ms": ms, "nbytes": nbytes, "streams": n_streams, "frames": n_frames, "seed": seed},
        "damaged_frames": {k: int((kind == v).sum()) for k, v in (("drop", 1), ("flip", 2), ("truncate", 3), ("garbage", 4))},
        "concealed_frames": int(o_concealed.sum()),
        "flip_survivors": int(((kind == 2) & ~o_concealed).sum()),     # bit flips the decoder cannot see (no CRC in LC3)
        "pcm_exact_fraction": float((diff == 0).mean()),
        "pcm_max_abs_diff": int(diff.max()),
    }
    rd = recovery_distance(o_clean, g_pcm, o_concealed)
    ro = recovery_distance(o_clean, o_pcm, o_concealed)
    # the engine's PCM may sit 1 LSB from the oracle's, which can move a frame across the "+-1 LSB of clean" line
    assert rd.size == ro.size and (rd.size == 0 or (rd != ro).mean() < 0.02), "recovery after concealment differs from the oracle's"
    rep["recovery_frames"] = {"runs": int(rd.size), "mean": float(rd.mean()) if rd.size else None,
                              "histogram": np.bincount(rd, minlength=9).tolist() if rd.size else []}
    if multi:                                 # the same damaged batch through the time-parallel entry point
        sf, fd = L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)
        ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(n_streams, fd, sf, nbytes), dtype=torch.uint8, device="cuda:0")
        dec = L.Lc3BatchDecoder(n_streams, fd, sf, ws, nbytes)
        scratch = torch.empty(dec.multi_scratch_bytes(n_frames), dtype=torch.uint8, device="cuda:0")
        pcm = torch.empty((n_streams, n_frames * dec.nf), dtype=torch.int16, device="cuda:0")
        status = torch.zeros((n_streams, n_frames), dtype=torch.int32, device="cuda:0")
        dec.decode_stream_frames(16, torch.from_numpy(damaged).to("cuda:0"), pcm, scratch,
                                 torch.from_numpy(lens).to("cuda:0"), status_out=status)
        m_pcm = pcm.cpu().numpy().reshape(n_streams, n_frames, dec.nf)
        assert np.array_equal(status.cpu().numpy(), g_status), "time-parallel path: concealed flags differ"
        assert np.array_equal(m_pcm, g_pcm), "time-parallel path: PCM differs from the frame-by-frame path"
        rep["time_parallel_identical"] = True
    return rep


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--fs", type=int, default=48000)
    ap.add_argument("--ms", type=float, default=10)
    ap.add_argument("--nbytes", type=int, default=150)
    ap.add_argument("--streams", type=int, default=2048)
    ap.add_argument("--frames", type=int, default=64)
    ap.add_argument("--seed", type=int, default=1)
    a = ap.parse_args()
    print(json.dumps(run(a.fs, a.ms if a.ms != 10 else 10, a.nbytes, a.streams, a.frames, a.seed)))


if __name__ == "__main__":
    main()
