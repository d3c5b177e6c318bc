"""Time-parallel decode (SURVEY.md 8f-1, lc3b_decode_stream_frames): many frames per stream in one call.

Contract: the call equals n_frames frame-by-frame calls - identical PCM (bit for bit: same arithmetic) and identical
per-stream state afterwards, so the two entry points can be interleaved.  Checked against the frame-by-frame GPU path
and (+-1 LSB) against the oracle, with LTPF transitions, lost and corrupted frames, 2- and 3-block LTPF histories.
"""
import numpy as np
import pytest

from common import assert_pcm_matches_oracle, corpus, gpu_decode

pytestmark = pytest.mark.gpu


def _decoder(fs, ms, S, nb):
    import torch

    import lc3_codec_b200 as L
    sf, fd = L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)
    ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(S, fd, sf, nb), dtype=torch.uint8, device="cuda:0")
    return L.Lc3BatchDecoder(S, fd, sf, ws, nb), ws


def _multi(dec, frames, lens=None):
    """frames [S, F, nb] -> pcm [S, F, nf] through one lc3b_decode_stream_frames call."""
    import torch
    S, F, nb = frames.shape
    scratch = torch.empty(dec.multi_scratch_bytes(F), dtype=torch.uint8, device="cuda:0")
    out = torch.zeros((S, F * dec.nf), dtype=torch.int16, device="cuda:0")
    st = torch.zeros((S, F), dtype=torch.int32, device="cuda:0")
    ln = None if lens is None else torch.from_numpy(np.ascontiguousarray(lens.astype(np.int32))).cuda()
    dec.decode_stream_frames(16, torch.from_numpy(np.ascontiguousarray(frames)).cuda(), out, scratch, ln, st)
    torch.cuda.synchronize()
    return out.cpu().numpy().reshape(S, F, dec.nf), st.cpu().numpy()


def _single(dec, frames, lens=None):
    import torch
    S, F, nb = frames.shape
    out = np.zeros((S, F, dec.nf), np.int16)
    for f in range(F):
        o = torch.zeros((S, dec.nf), dtype=torch.int16, device="cuda:0")
        ln = None if lens is None else torch.from_numpy(np.ascontiguousarray(lens[:, f].astype(np.int32))).cuda()
        dec.decode_frames(16, torch.from_numpy(np.ascontiguousarray(frames[:, f])).cuda(), o, ln)
        out[:, f] = o.cpu().numpy()
    return out


@pytest.mark.parametrize("fs,ms,nbytes", [(48000, 10, 150), (16000, 7.5, 30), (48000, 10, 60), (32000, 7.5, 45), (24000, 10, 40)])
def test_multi_equals_frame_by_frame_and_oracle(fs, ms, nbytes):
    _, frames = corpus(fs, ms, nbytes, 48, 40)
    dec, _ws = _decoder(fs, ms, 48, nbytes)
    got, status = _multi(dec, frames)
    ref = gpu_decode(fs, ms, frames, trace=False)[0]
    assert np.array_equal(got, ref), "time-parallel PCM differs from the frame-by-frame path"
    assert_pcm_matches_oracle(got, fs, ms, frames)
    assert status.shape == (48, 40)


def test_multi_with_lost_and_corrupt_frames():
    """Concealment along time: dropped frames, long runs, loss at the start, bit flips; LTPF active around the losses."""
    _, frames = corpus(48000, 10, 60, 64, 48)
    frames = frames.copy()
    S, F, nb = frames.shape
    rng = np.random.default_rng(5)
    lens = np.full((S, F), nb, np.int32)
    lens[rng.random((S, F)) < 0.10] = 0
    lens[3, 8:22] = 0
    lens[4, 0:3] = 0
    lens[5, F - 2:] = 0
    for s, f in np.argwhere(rng.random((S, F)) < 0.08):
        frames[s, f, rng.integers(0, nb)] ^= 1 << int(rng.integers(0, 8))
    dec, _ws = _decoder(48000, 10, S, nb)
    got, status = _multi(dec, frames, lens)
    ref_pcm, ref_tr, _, _, ref_status = gpu_decode(48000, 10, frames, lens)
    assert np.array_equal(status, ref_status)
    assert np.array_equal(got, ref_pcm)
    assert status.mean() > 0.05


def test_multi_and_single_calls_interleave():
    """State hand-back: multi(13 frames) + 5 single calls + multi(22 frames) == 40 single calls, LTPF and PLC state included."""
    fs, ms, nbytes = 16000, 7.5, 30
    _, frames = corpus(fs, ms, nbytes, 40, 40)
    frames = frames.copy()
    lens = np.full(frames.shape[:2], nbytes, np.int32)
    lens[7, 11:15] = 0                                   # a loss that straddles the first hand-over
    lens[9, 17:19] = 0
    dec, _ws = _decoder(fs, ms, 40, nbytes)
    a, _ = _multi(dec, frames[:, :13], lens[:, :13])
    b = _single(dec, frames[:, 13:18], lens[:, 13:18])
    c, _ = _multi(dec, frames[:, 18:], lens[:, 18:])
    got = np.concatenate([a, b, c], axis=1)
    ref = gpu_decode(fs, ms, frames, lens, trace=False)[0]
    assert np.array_equal(got, ref)


def test_multi_file_shape_few_streams_many_frames():
    """The workload the path exists for: 2 channels x 600 frames in one call."""
    _, frames = corpus(48000, 10, 150, 2, 600)
    dec, _ws = _decoder(48000, 10, 2, 150)
    got, _ = _multi(dec, frames)
    assert_pcm_matches_oracle(got, 48000, 10, frames)
