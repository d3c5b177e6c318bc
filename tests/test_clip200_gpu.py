"""Parity on the contract's corpus: SURVEY.md 8d clips of 200 frames per stream (2 s / 1.5 s of audio).

Short clips under-test exactly the data-dependent kernels: the noise class spends a third of a 12-frame clip in its
two 100 ms silent gaps, a 6-frame clip never leaves them.  At 200 frames the gaps are 10 % of the stream and broadband
noise frames (highest lastnz, most escapes and residual bits), complete sine sweeps and every voiced / unvoiced
transition of the speech class are decoded with the state a real stream carries.  Oracle cost: seconds.

  C1   48 kHz / 10 ms / 150 B   decode: side info + integer spectrum + shaped spectrum bit exact, PCM +-1 LSB
  C3   16 kHz / 7.5 ms / 30 B   same (LTPF and TNS active, 3-block histories)
  44.1 kHz / 7.5 ms / 90, 60 B  same (at 60 B the post filter is on: l_den = 11 with the truncated 48 k tables)
  C2   48 kHz / 10 ms / 120 B   encode: bytes identical to the oracle encoder's on every frame
  time-parallel decode of whole 200-frame clips in ONE call (the examples/decode.rs shape)
Run on the B200 box: python -m pytest tests -m gpu
"""
import numpy as np
import pytest

from common import assert_encoder_parity, assert_parity, assert_pcm_matches_oracle, corpus_clip

pytestmark = pytest.mark.gpu


def test_c1_48k_10ms_150B_200_frames():
    _, frames = corpus_clip(48000, 10, 150, 192)
    assert frames.shape == (192, 200, 150)
    stats = assert_parity(48000, 10, frames)
    # the corpus statistics the judge measured for 8d clips (mean lastnz 362, 2.8 % near-empty frames, lsb_mode 7.4 %)
    assert stats["mean_lastnz"] >= 340 and stats["near_empty"] <= 0.08 and stats["lsb_mode"] >= 0.04, stats
    assert stats["concealed"] <= 0.001 and stats["tns"] > 0.2, stats


def test_c3_16k_7p5ms_30B_200_frames():
    _, frames = corpus_clip(16000, 7.5, 30, 192)
    stats = assert_parity(16000, 7.5, frames)
    assert stats["ltpf_active"] > 0.05 and stats["tns"] > 0.1, stats


@pytest.mark.parametrize("nbytes", [90, 60])
def test_44k1_7p5ms_200_frames(nbytes):
    _, frames = corpus_clip(44100, 7.5, nbytes, 96)
    stats = assert_parity(44100, 7.5, frames)
    assert (stats["ltpf_active"] > 0.2) == (nbytes == 60), stats     # 90 B: 960 scaled bits >= 880, gain table row (0.0, 0)


def test_c2_encode_48k_10ms_120B_200_frames():
    assert assert_encoder_parity(48000, 10, 120, 96, 0, clip=True) == 1.0


def test_encode_16k_7p5ms_30B_200_frames():
    assert assert_encoder_parity(16000, 7.5, 30, 96, 0, clip=True) == 1.0


@pytest.mark.parametrize("fs,ms,nbytes", [(48000, 10, 150), (16000, 7.5, 30)])
def test_time_parallel_whole_clip(fs, ms, nbytes):
    """One lc3b_decode_stream_frames call over the full 200-frame clips of 96 streams."""
    import torch

    import lc3_codec_b200 as L
    _, frames = corpus_clip(fs, ms, nbytes, 192)
    frames = frames[:96]
    S, F, nb = frames.shape
    sf, fd = L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)
    ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(S, fd, sf, nb), dtype=torch.uint8, device="cuda:0")
    dec = L.Lc3BatchDecoder(S, fd, sf, ws, nb)
    scratch = torch.empty(dec.multi_scratch_bytes(F), dtype=torch.uint8, device="cuda:0")
    out = torch.zeros((S, F * dec.nf), dtype=torch.int16, device="cuda:0")
    dec.decode_stream_frames(16, torch.from_numpy(np.ascontiguousarray(frames)).cuda(), out, scratch)
    torch.cuda.synchronize()
    assert_pcm_matches_oracle(out.cpu().numpy().reshape(S, F, dec.nf), fs, ms, frames)
