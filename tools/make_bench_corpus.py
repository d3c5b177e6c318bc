#!/usr/bin/env python3
"""Dev-time generator of the bitstream fixtures bench.py decodes (SURVEY.md section 8d corpus).

Every stream is a 200-frame clip of tools/corpus.py (classes sweep / noise / speech-like), encoded from frame 0 by
the ORACLE encoder (the reference encoder cannot run here) so that the encoder state is the clip's own; the fixture
keeps N_FRAMES consecutive frames of every stream starting at a per-stream offset drawn from [10, 200 - N_FRAMES]
(the first 10 frames are the encoder's start-up and are excluded, as SURVEY 8d excludes them from statistics).  The
offsets are spread over the whole clip, so the fixture samples every part of the sweep, the noise class's two silent
gaps at their real 10 % duty and the voiced / unvoiced alternation of the speech class.

  tests/golden/bench_c1_frames_{0,1}.npy  [1024, 8, 150] u8 in two halves of 512 streams (tools.corpus.load_bench_c1_frames)
                                        48 kHz / 10 ms / 150 B   (BASELINE configs 1 and 5)
  tests/golden/bench_c1_stats.json      corpus statistics from the oracle decoder (mean lastnz, near-empty, lsb_mode ...)
  tests/golden/bench_mixed_8k_*.npy     8 kHz bitstreams for the mixed-rate bench (no 8 kHz encoder in the reference)

bench.py tiles these streams up to the batch size, so the product benchmark itself never executes oracle code.
Usage: python tools/make_bench_corpus.py
"""
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from oracle import pyoracle as O  # noqa: E402
from tools.corpus import (BENCH_C1_PARTS, CLIP_FRAMES, CLIP_SKIP as SKIP, GOLDEN, clip_offsets, make_pcm,  # noqa: E402
                          take_window)

N_FRAMES = 8


def stats_of(frames: np.ndarray, fs: int, ms: float) -> dict:
    """Statistics of a [S, F, nbytes] bitstream set from the oracle decoder's side information."""
    _, tr, x, _ = O.decode_streams(frames, fs, ms, trace=True)
    ok = tr[..., O.TR["OK"]] == 1
    lastnz = tr[..., O.TR["LASTNZ"]][ok]
    return {"streams": int(frames.shape[0]), "frames_per_stream": int(frames.shape[1]),
            "mean_lastnz": float(lastnz.mean()), "near_empty_frac": float((lastnz <= 16).mean()),
            "lsb_mode_frac": float(tr[..., O.TR["LSB_MODE"]][ok].mean()),
            "mean_nonzero_lines": float((x[ok] != 0).sum(-1).mean()),
            "concealed_frac": float(1.0 - ok.mean()),
            "tns_active_frac": float((tr[..., O.TR["RC_ORDER0"]][ok] > 0).mean()),
            "ltpf_active_frac": float(tr[..., O.TR["LTPF_ACTIVE"]][ok].mean())}


def main():
    n_streams = 1024
    pcm = make_pcm(n_streams, CLIP_FRAMES, 48000, 480)
    full = O.encode_streams(pcm, 48000, 10, 150)
    off = clip_offsets(n_streams, N_FRAMES)
    frames = take_window(full, off, N_FRAMES)
    half = n_streams // len(BENCH_C1_PARTS)
    for k, name in enumerate(BENCH_C1_PARTS):
        out = GOLDEN / name
        np.save(out, frames[k * half:(k + 1) * half])
        print(out, out.stat().st_size)
    st = stats_of(frames, 48000, 10)
    st.update({"clip_frames": CLIP_FRAMES, "first_frame_min": int(off.min()), "first_frame_max": int(off.max()),
               "whole_clip_frames_10_199": stats_of(full[:192, SKIP:], 48000, 10),
               "source": "tools/make_bench_corpus.py: 200-frame clips (SURVEY 8d), oracle encoder, 8 consecutive frames "
                         "per stream at a per-stream offset in [10, 192]"})
    (ROOT / "tests" / "golden" / "bench_c1_stats.json").write_text(json.dumps(st, indent=1) + "\n")
    print(frames.shape, frames.dtype)
    print(json.dumps(st, indent=1))

    # 8 kHz bitstreams for the mixed-rate bench (BASELINE config 4): the reference encoder (and therefore the GPU
    # encoder) cannot be constructed at 8 kHz, so these come from the oracle encoder's spec-following 8 kHz path.
    for ms, nb, nf in ((7.5, 20, 60), (10, 26, 80)):
        pcm8 = make_pcm(512, CLIP_FRAMES, 8000, nf)
        fr8 = take_window(O.encode_streams(pcm8, 8000, ms, nb), clip_offsets(512, N_FRAMES), N_FRAMES)
        out8 = ROOT / "tests" / "golden" / f"bench_mixed_8k_{str(ms).replace('.', 'p')}ms.npy"
        np.save(out8, fr8)
        print(out8, fr8.shape, out8.stat().st_size)


if __name__ == "__main__":
    main()
