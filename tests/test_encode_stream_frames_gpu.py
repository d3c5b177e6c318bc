"""Time-parallel encode (lc3b_encode_stream_frames): many consecutive frames of every stream in one call.

Contract: the call equals n_frames frame-by-frame lc3b_encode_frames calls with the same nbytes - identical bytes and
identical per-stream state afterwards, so the two entry points can be interleaved.  Checked byte for byte against the
frame-by-frame GPU path over every encoder configuration, at rates that switch the attack detector and the LTPF on and
off, and through the encoder gate against the oracle.
"""
import ctypes as C

import numpy as np
import pytest

from common import corpus, corpus_clip, encoder_gate, gpu_encode

pytestmark = pytest.mark.gpu


def _encoder(fs, ms, S, nb):
    import torch

    import lc3_codec_b200 as L
    sf, fd = L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)
    ws = torch.empty(L.Lc3BatchEncoder.calc_working_buffer_lengths(S, fd, sf, nb), dtype=torch.uint8, device="cuda:0")
    return L.Lc3BatchEncoder(S, fd, sf, ws, nb)


def _multi(enc, pcm, nbytes):
    """pcm [S, F, nf] -> bytes [S, F, nbytes] through one lc3b_encode_stream_frames call."""
    import torch
    S, F, nf = pcm.shape
    scratch = torch.empty(enc.multi_scratch_bytes(F), dtype=torch.uint8, device="cuda:0")
    out = torch.zeros((S, F, nbytes), dtype=torch.uint8, device="cuda:0")
    enc.encode_stream_frames(torch.from_numpy(np.ascontiguousarray(pcm.reshape(S, F * nf))).cuda(), out, scratch)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def _single(enc, pcm, nbytes):
    import torch
    S, F, nf = pcm.shape
    out = np.zeros((S, F, nbytes), np.uint8)
    for f in range(F):
        y = torch.zeros((S, nbytes), dtype=torch.uint8, device="cuda:0")
        enc.encode_frames(torch.from_numpy(np.ascontiguousarray(pcm[:, f])).cuda(), y)
        out[:, f] = y.cpu().numpy()
    return out


# every encoder configuration; the attack detector is on at 48 kHz / 10 ms from 100 B, at 32 kHz / 7.5 ms in [61, 150),
# at 44.1-48 kHz / 7.5 ms in [75, 150); the LTPF gain region ends at 560 + 80 fs_ind bits per 10 ms (110 B at 48 kHz)
CASES = [(16000, 10, 20), (16000, 7.5, 30), (24000, 10, 40), (24000, 7.5, 45), (32000, 10, 90), (32000, 7.5, 70),
         (44100, 10, 100), (44100, 7.5, 400), (48000, 10, 60), (48000, 10, 120), (48000, 7.5, 75), (48000, 10, 400)]


@pytest.mark.parametrize("fs,ms,nbytes", CASES)
def test_one_call_equals_frame_by_frame(fs, ms, nbytes):
    S, F = 48, 40
    pcm, o_frames = corpus(fs, ms, nbytes, S, F)
    g = _multi(_encoder(fs, ms, S, nbytes), pcm, nbytes)
    ref = gpu_encode(fs, ms, pcm, nbytes)
    bad = np.argwhere((g != ref).any(-1))
    assert bad.size == 0, f"{len(bad)} frames differ from the frame-by-frame path, first (stream, frame) {bad[:5].tolist()}"
    encoder_gate(pcm, o_frames, g, fs, ms)


@pytest.mark.parametrize("fs,ms,nbytes", [(48000, 10, 120), (32000, 7.5, 70)])
def test_state_hand_back_between_entry_points(fs, ms, nbytes):
    S, F = 24, 40
    pcm, _ = corpus(fs, ms, nbytes, S, F)
    ref = gpu_encode(fs, ms, pcm, nbytes)
    enc = _encoder(fs, ms, S, nbytes)
    got = np.concatenate([_multi(enc, pcm[:, :13], nbytes), _single(enc, pcm[:, 13:18], nbytes),
                          _multi(enc, pcm[:, 18:], nbytes)], axis=1)
    assert np.array_equal(got, ref)
    # one frame per call through the time-parallel entry point is the frame-by-frame call
    enc1, enc2 = _encoder(fs, ms, S, nbytes), _encoder(fs, ms, S, nbytes)
    for f in range(3):
        assert np.array_equal(_multi(enc1, pcm[:, f:f + 1], nbytes), _single(enc2, pcm[:, f:f + 1], nbytes))


def test_range_coder_kernel_path_over_12288_units():
    """64 SURVEY clips x 200 frames = 12 800 units: the bitstream stage runs the thread-per-frame range coder kernel
    (the 48-stream cases above run it inline)."""
    fs, ms, nbytes, S = 48000, 10, 150, 64
    pcm, o_frames = corpus_clip(fs, ms, nbytes, S)
    g = _multi(_encoder(fs, ms, S, nbytes), pcm, nbytes)
    assert np.array_equal(g, gpu_encode(fs, ms, pcm, nbytes))
    encoder_gate(pcm, o_frames, g, fs, ms)


def test_graph_mode_on_and_off_give_the_same_bytes():
    fs, ms, nbytes, S, F = 48000, 10, 120, 16, 24
    pcm, _ = corpus(fs, ms, nbytes, S, F)
    out = []
    for graph in (True, False):
        enc = _encoder(fs, ms, S, nbytes)
        enc.set_graph_mode(graph)
        out.append(np.concatenate([_multi(enc, pcm[:, :12], nbytes), _multi(enc, pcm[:, 12:], nbytes)], axis=1))
    assert np.array_equal(out[0], out[1])
    assert np.array_equal(out[0], gpu_encode(fs, ms, pcm, nbytes))


def test_file_shape_two_channels_600_frames():
    fs, ms, nbytes, S, F = 48000, 10, 150, 2, 600
    pcm, o_frames = corpus(fs, ms, nbytes, S, F)
    g = _multi(_encoder(fs, ms, S, nbytes), pcm, nbytes)
    assert np.array_equal(g, gpu_encode(fs, ms, pcm, nbytes))
    encoder_gate(pcm, o_frames, g, fs, ms)


def test_argument_errors():
    import torch

    import lc3_codec_b200 as L
    lib = L.lib()
    S, nb, F = 4, 120, 3
    enc = _encoder(48000, 10, S, nb)
    h = enc._h
    need = enc.multi_scratch_bytes(F)
    scratch = torch.empty(need + 256, dtype=torch.uint8, device="cuda:0")
    pcm = torch.zeros((S, F * 480), dtype=torch.int16, device="cuda:0")
    out = torch.zeros((S, F, nb), dtype=torch.uint8, device="cuda:0")
    P = lambda t, off=0: C.c_void_p(t.data_ptr() + off)   # noqa: E731
    sp, pp, op = P(scratch), P(pcm), P(out)

    def call(h=h, pcm=pp, n_frames=F, out=op, nbytes=nb, stride=nb, scratch=sp, scratch_bytes=need):
        return lib.lc3b_encode_stream_frames(h, pcm, n_frames, out, nbytes, stride, scratch, scratch_bytes, None)

    assert call() == 0
    torch.cuda.synchronize()
    assert call(h=None) == 2
    assert call(pcm=None) == 2 and call(out=None) == 2 and call(scratch=None) == 2
    assert call(nbytes=19, stride=19) == 2                         # below the side information
    assert call(nbytes=nb + 1, stride=nb + 1) == 2                 # above the handle's max_nbytes
    assert call(stride=nb - 1) == 2                                # nbytes > frame_stride
    assert call(n_frames=0) == 2 and call(n_frames=-1) == 2
    assert call(n_frames=(2 ** 31) // S + 1) == 2                  # n_streams * n_frames beyond an int
    assert call(scratch_bytes=need - 1) == 4                       # short by one byte
    assert call(scratch=P(scratch, 1)) == 4                        # misaligned
    n = C.c_size_t(0)
    assert lib.lc3b_encoder_multi_scratch_bytes(h, 0, C.byref(n)) == 2
    assert lib.lc3b_encoder_multi_scratch_bytes(h, (2 ** 31) // S + 1, C.byref(n)) == 2
    assert lib.lc3b_encoder_multi_scratch_bytes(h, F, None) == 2
    assert lib.lc3b_encoder_multi_scratch_bytes(h, F, C.byref(n)) == 0 and n.value == need
    with pytest.raises(L.Lc3bError):                               # the Python mirror checks shapes first
        enc.encode_stream_frames(pcm[:, :-1], out, scratch)
    with pytest.raises(L.Lc3bError):
        enc.encode_stream_frames(pcm, out, scratch[:need - 1])
