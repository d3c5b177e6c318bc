"""The committed bench fixtures are the SURVEY.md 8d corpus: 200-frame clips, 8 consecutive frames per stream.

Checks (oracle only, no GPU): the statistics file matches what the oracle decoder sees in the fixture, the statistics
meet the bar the round-1 review set (mean lastnz >= 350, near-empty frames <= 5 %), and the fixture is reproducible
from tools/make_bench_corpus.py's recipe (first 24 streams regenerated here).
"""
import json

import numpy as np

from conftest import GOLDEN
from oracle import pyoracle as O
from tools.corpus import CLIP_FRAMES, clip_offsets, load_bench_c1_frames, make_pcm, take_window
from tools.make_bench_corpus import N_FRAMES, stats_of


def test_fixture_statistics():
    frames = load_bench_c1_frames()
    assert frames.shape == (1024, N_FRAMES, 150) and frames.dtype == np.uint8
    doc = json.loads((GOLDEN / "bench_c1_stats.json").read_text())
    st = stats_of(frames, 48000, 10)
    for k, v in st.items():
        assert doc[k] == v, (k, doc[k], v)
    assert st["mean_lastnz"] >= 350 and st["near_empty_frac"] <= 0.05 and st["lsb_mode_frac"] >= 0.05, st
    assert st["concealed_frac"] == 0.0
    whole = doc["whole_clip_frames_10_199"]                  # the window sample is representative of the whole clips
    assert abs(whole["mean_lastnz"] - st["mean_lastnz"]) < 10 and abs(whole["near_empty_frac"] - st["near_empty_frac"]) < 0.01


def test_fixture_is_reproducible():
    frames = load_bench_c1_frames()
    n = 24
    full = O.encode_streams(make_pcm(n, CLIP_FRAMES, 48000, 480), 48000, 10, 150)
    off = clip_offsets(n, N_FRAMES)
    assert off.min() >= 10 and off.max() <= CLIP_FRAMES - N_FRAMES
    assert np.array_equal(take_window(full, off, N_FRAMES), frames[:n])
    fr8 = np.load(GOLDEN / "bench_mixed_8k_10ms.npy")
    full8 = O.encode_streams(make_pcm(n, CLIP_FRAMES, 8000, 80), 8000, 10, 26)
    assert np.array_equal(take_window(full8, clip_offsets(n, N_FRAMES), N_FRAMES), fr8[:n])
