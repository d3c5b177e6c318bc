"""Subset calls and stream resets (lc3b_decode_frames_subset, lc3b_encode_frames_subset, lc3b_*_reset_streams).

Contract: a stream's PCM / status / spectrum (decoder) or bytes (encoder) and its state after any mix of subset calls,
full calls, time-parallel calls and resets are exactly what the stream gets when it runs the same frame sequence in a
handle of its own.  The reference is a "lockstep" handle: one row per stream sequence, row v of frame-by-frame call k
carries the k-th frame that sequence received.  A reset starts a new sequence on the same stream id.  Only the frames a
sequence actually received are compared.
"""
import ctypes as C

import numpy as np
import pytest

from common import corpus, encoder_gate, gpu_decode, gpu_encode
from tools.corpus import make_pcm

pytestmark = pytest.mark.gpu


def _decoder(fs, ms, S, nb, dequant_mode=0, synth_mode=0, graph=None, split=None):
    import torch

    import lc3_codec_b200 as L
    sf, fd = L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)
    ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(S, fd, sf, nb), dtype=torch.uint8, device="cuda:0")
    dec = L.Lc3BatchDecoder(S, fd, sf, ws, nb)
    dec.set_dequant_mode(dequant_mode)
    dec.set_synth_mode(synth_mode)
    if graph is not None:
        dec.set_graph_mode(graph)
    if split is not None:
        dec.set_split(split)
    return dec


def _encoder(fs, ms, S, nb, graph=None):
    import torch

    import lc3_codec_b200 as L
    sf, fd = L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)
    ws = torch.empty(L.Lc3BatchEncoder.calc_working_buffer_lengths(S, fd, sf, nb), dtype=torch.uint8, device="cuda:0")
    enc = L.Lc3BatchEncoder(S, fd, sf, ws, nb)
    if graph is not None:
        enc.set_graph_mode(graph)
    return enc


class Book:
    """Which frame sequence each stream id runs and how many of its frames it has had."""

    def __init__(self, S):
        self.seq = list(range(S))
        self.cnt = [0] * S
        self.n_seq = S

    def take(self, ids):
        vk = [(self.seq[s], self.cnt[s]) for s in ids]
        for s in ids:
            self.cnt[s] += 1
        return vk

    def reset(self, ids):
        for s in ids:
            self.seq[s] = self.n_seq
            self.n_seq += 1
            self.cnt[s] = 0


def _schedule(S, P, rng, min_rows=1):
    """P id lists: random subsets in random order, with an empty call, a single stream and all streams among them."""
    out = []
    for p in range(P):
        if p == 3:
            n = 0
        elif p == 5:
            n = 1
        elif p == 7:
            n = S
        else:
            n = int(rng.integers(min_rows, S + 1))
        out.append(rng.permutation(S)[:n].astype(np.int32))
    return out


def _decode_rows(dec, ids, frames, lens):
    import torch
    n = len(ids)
    out = torch.full((n, dec.nf), 12345, dtype=torch.int16, device="cuda:0")
    st = torch.full((n,), 7, dtype=torch.int32, device="cuda:0")
    ln = None if lens is None else torch.from_numpy(np.ascontiguousarray(lens, dtype=np.int32)).cuda()
    dec.decode_frames_subset(16, ids, torch.from_numpy(np.ascontiguousarray(frames)).cuda(), out, ln, status_out=st)
    return out.cpu().numpy(), st.cpu().numpy()


def _run_decoder_schedule(dec, S, sched, frames, lens=None, resets=None):
    """Runs the schedule on `dec`; returns Book and {(seq, k): (pcm, status)}."""
    book, got = Book(S), {}
    for p, ids in enumerate(sched):
        if resets and p in resets:
            dec.reset_streams(resets[p])
            book.reset(resets[p])
        vk = book.take(ids)
        rows = np.array([frames[v, k] for v, k in vk], np.uint8).reshape(len(ids), frames.shape[2])
        rl = None if lens is None else np.array([lens[v, k] for v, k in vk], np.int32)
        pcm, st = _decode_rows(dec, ids, rows, rl)
        if len(ids) == 0:
            assert pcm.shape[0] == 0
        for i, key in enumerate(vk):
            got[key] = (pcm[i], st[i])
    return book, got


def _check_decoder(book, got, ref, spectrum_now, S):
    r_pcm, _tr, _x, r_sp, r_status = ref
    for (v, k), (pcm, st) in got.items():
        assert np.array_equal(pcm, r_pcm[v, k]), f"PCM of sequence {v} frame {k} differs from the lockstep handle"
        assert st == r_status[v, k], f"status of sequence {v} frame {k}"
    for s in range(S):                                            # the spectrum the stream's last frame left
        v, n = book.seq[s], book.cnt[s]
        want = r_sp[v, n - 1] if n else np.zeros_like(r_sp[0, 0])
        assert np.array_equal(spectrum_now[s].view(np.uint32), want.view(np.uint32)), f"spectrum of stream {s}"


DEC_CASES = [(48000, 10, 150, False), (16000, 7.5, 30, False), (24000, 10, 40, True)]


@pytest.mark.parametrize("fs,ms,nbytes,lossy", DEC_CASES)
def test_decoder_schedule_equals_lockstep(fs, ms, nbytes, lossy):
    """48 kHz / 150 B has lsb_mode frames; 16 kHz / 30 B runs the post filter (ltpf_kernel); the lossy case feeds lost
    (length 0) and garbage frames, so streams are concealed."""
    S, P = 96, 30
    rng = np.random.default_rng(11)
    _, frames = corpus(fs, ms, nbytes, S, P)
    frames = frames.copy()
    lens = None
    if lossy:
        lens = np.full((S, P), nbytes, np.int32)
        lens[rng.random((S, P)) < 0.1] = 0
        bad = rng.random((S, P)) < 0.1
        frames[bad] = rng.integers(0, 256, (int(bad.sum()), nbytes), dtype=np.uint8)
    sched = _schedule(S, P, rng)
    dec = _decoder(fs, ms, S, nbytes)
    book, got = _run_decoder_schedule(dec, S, sched, frames, lens)
    ref = gpu_decode(fs, ms, frames, lens)
    _check_decoder(book, got, ref, dec.spectrum().cpu().numpy(), S)
    if lossy:
        assert any(st == 1 for _, st in got.values())


@pytest.mark.parametrize("opts", [dict(dequant_mode=1), dict(dequant_mode=2), dict(synth_mode=1), dict(synth_mode=0),
                                  dict(graph=True), dict(graph=False)])
def test_decoder_every_kernel_choice(opts):
    fs, ms, nbytes, S, P = 16000, 7.5, 30, 96, 16
    rng = np.random.default_rng(5)
    _, frames = corpus(fs, ms, nbytes, S, P)
    sched = _schedule(S, P, rng)
    dec = _decoder(fs, ms, S, nbytes, **opts)
    book, got = _run_decoder_schedule(dec, S, sched, frames)
    _check_decoder(book, got, gpu_decode(fs, ms, frames), dec.spectrum().cpu().numpy(), S)


def test_decoder_split_sub_batches():
    """set_split(4): calls of 512 rows and more are cut into sub-batches; the state pointers stay at the handle's base."""
    fs, ms, nbytes, S, P = 48000, 10, 150, 640, 6
    rng = np.random.default_rng(9)
    _, frames = corpus(fs, ms, nbytes, S, P)
    sched = [rng.permutation(S)[:n].astype(np.int32) for n in (640, 600, 512, 100, 531, 640)]
    for graph in (False, True):
        dec = _decoder(fs, ms, S, nbytes, dequant_mode=2, split=4)   # the warp-per-frame dequantisation is never split
        dec.set_graph_mode(graph)
        book, got = _run_decoder_schedule(dec, S, sched, frames)
        _check_decoder(book, got, gpu_decode(fs, ms, frames), dec.spectrum().cpu().numpy(), S)


def test_decoder_subset_then_full_then_time_parallel():
    import torch
    fs, ms, nbytes, S = 16000, 7.5, 30, 96
    rng = np.random.default_rng(3)
    P, FULL, MULTI = 10, 3, 5
    _, frames = corpus(fs, ms, nbytes, S, P + FULL + MULTI)
    dec = _decoder(fs, ms, S, nbytes)
    book, got = _run_decoder_schedule(dec, S, _schedule(S, P, rng), frames)
    ids = np.arange(S)
    for _ in range(FULL):                                         # full calls: row s is stream s
        vk = book.take(ids)
        rows = np.array([frames[v, k] for v, k in vk])
        out = torch.zeros((S, dec.nf), dtype=torch.int16, device="cuda:0")
        st = torch.zeros(S, dtype=torch.int32, device="cuda:0")
        dec.decode_frames(16, torch.from_numpy(rows).cuda(), out, status_out=st)
        for i, key in enumerate(vk):
            got[key] = (out[i].cpu().numpy(), int(st[i]))
    start = [book.cnt[s] for s in range(S)]
    block = np.stack([frames[s, start[s]:start[s] + MULTI] for s in range(S)])
    scratch = torch.empty(dec.multi_scratch_bytes(MULTI), dtype=torch.uint8, device="cuda:0")
    out = torch.zeros((S, MULTI * dec.nf), dtype=torch.int16, device="cuda:0")
    st = torch.zeros((S, MULTI), dtype=torch.int32, device="cuda:0")
    dec.decode_stream_frames(16, torch.from_numpy(np.ascontiguousarray(block)).cuda(), out, scratch, status_out=st)
    out, st = out.cpu().numpy().reshape(S, MULTI, dec.nf), st.cpu().numpy()
    for f in range(MULTI):
        for i, key in enumerate(book.take(ids)):
            got[key] = (out[i, f], st[i, f])
    _check_decoder(book, got, gpu_decode(fs, ms, frames), dec.spectrum().cpu().numpy(), S)


@pytest.mark.parametrize("fs,ms,nbytes", [(16000, 7.5, 30), (48000, 10, 150)])
def test_decoder_reset_streams(fs, ms, nbytes):
    """Reset streams continue like a freshly initialised handle fed the frames from that point; the others are untouched."""
    S, P = 96, 20
    rng = np.random.default_rng(21)
    resets = {6: rng.permutation(S)[:30].astype(np.int32), 13: rng.permutation(S)[:50].astype(np.int32), 15: np.zeros(0, np.int32)}
    V = S + 80
    _, frames = corpus(fs, ms, nbytes, V, P)
    dec = _decoder(fs, ms, S, nbytes)
    book, got = _run_decoder_schedule(dec, S, _schedule(S, P, rng), frames, resets=resets)
    assert book.n_seq == V
    _check_decoder(book, got, gpu_decode(fs, ms, frames), dec.spectrum().cpu().numpy(), S)


def test_decoder_rejects_bad_id_lists_and_enqueues_nothing():
    import torch

    import lc3_codec_b200 as L
    fs, ms, nbytes, S = 48000, 10, 150, 32
    _, frames = corpus(fs, ms, nbytes, S, 2)
    dec = _decoder(fs, ms, S, nbytes)
    lib = L.lib()
    fr = torch.from_numpy(np.ascontiguousarray(frames[:, 0])).cuda()
    out = torch.full((S, dec.nf), 777, dtype=torch.int16, device="cuda:0")
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(ids, n):
        arr = None if ids is None else np.ascontiguousarray(ids, dtype=np.int32)
        p = None if arr is None else C.c_void_p(arr.ctypes.data)
        return lib.lc3b_decode_frames_subset(dec._h, 16, p, n, C.c_void_p(fr.data_ptr()), None, nbytes, nbytes,
                                             C.c_void_p(out.data_ptr()), dec.nf, None, stream)

    assert call(None, 4) == 2                                     # null ids
    assert call([0, 1], -1) == 2
    assert call(np.arange(S + 1), S + 1) == 2                     # more rows than streams
    assert call([0, S], 2) == 2                                   # out of range
    assert call([-1, 0], 2) == 2
    assert call([3, 5, 3], 3) == 2                                # listed twice
    assert call([0, 1], 2) == 0 and call([], 0) == 0               # a valid list, then an empty call
    assert lib.lc3b_decoder_reset_streams(dec._h, None, 1, stream) == 2
    arr = np.array([2, 2], np.int32)
    assert lib.lc3b_decoder_reset_streams(dec._h, C.c_void_p(arr.ctypes.data), 2, stream) == 2
    with pytest.raises(L.Lc3DecoderError):
        dec.decode_frames_subset(8, [0], fr[:1], out[:1])
    with pytest.raises(L.Lc3bError):
        dec.decode_frames_subset(16, [0, 1], fr[:1], out[:1])     # rows do not match the id list
    torch.cuda.synchronize()
    # nothing but rows 0, 1 of the one valid call was written, and only streams 0 and 1 moved on
    assert (out[2:].cpu().numpy() == 777).all()
    rows = frames[:, 0].copy()
    rows[:2] = frames[:2, 1]                                      # streams 0 and 1 are one frame ahead
    out2 = torch.zeros((S, dec.nf), dtype=torch.int16, device="cuda:0")
    dec.decode_frames(16, torch.from_numpy(rows).cuda(), out2)
    ref = gpu_decode(fs, ms, frames, trace=False)[0]
    assert np.array_equal(out2.cpu().numpy()[2:], ref[2:, 0])
    assert np.array_equal(out2.cpu().numpy()[:2], ref[:2, 1])
    # the id list may also come as a CPU int32 tensor or a numpy array
    dec.decode_frames_subset(16, torch.tensor([4, 9], dtype=torch.int32), fr[:2], out[:2])
    dec.reset_streams(np.array([4, 9]))


# ---------------------------------------------------------------------------------------------------------- encoder
def _run_encoder_schedule(enc, S, sched, pcm, nbytes, resets=None):
    import torch
    book, got = Book(S), {}
    for p, ids in enumerate(sched):
        if resets and p in resets:
            enc.reset_streams(resets[p])
            book.reset(resets[p])
        vk = book.take(ids)
        rows = np.array([pcm[v, k] for v, k in vk], np.int16).reshape(len(ids), pcm.shape[2])
        out = torch.zeros((len(ids), nbytes), dtype=torch.uint8, device="cuda:0")
        enc.encode_frames_subset(ids, torch.from_numpy(rows).cuda(), out)
        out = out.cpu().numpy()
        for i, key in enumerate(vk):
            got[key] = out[i]
    return book, got


def _check_encoder(got, ref):
    for (v, k), b in got.items():
        assert np.array_equal(b, ref[v, k]), f"bytes of sequence {v} frame {k} differ from the lockstep handle"


# a spread of the time-parallel encoder's CASES: attack detector on (48 kHz / 10 ms / 120 B, 32 kHz / 7.5 ms / 70 B) and
# off, the LTPF region (16-24 kHz at low rates), 7.5 ms
ENC_CASES = [(16000, 7.5, 30), (24000, 10, 40), (32000, 7.5, 70), (48000, 10, 120), (48000, 10, 60), (44100, 7.5, 400)]


@pytest.mark.parametrize("fs,ms,nbytes", ENC_CASES)
def test_encoder_schedule_equals_lockstep(fs, ms, nbytes):
    S, P = 96, 30
    rng = np.random.default_rng(17)
    pcm, _ = corpus(fs, ms, nbytes, S, P)
    enc = _encoder(fs, ms, S, nbytes)
    _, got = _run_encoder_schedule(enc, S, _schedule(S, P, rng), pcm, nbytes)
    _check_encoder(got, gpu_encode(fs, ms, pcm, nbytes))


@pytest.mark.parametrize("graph", [False, True])
def test_encoder_graph_modes_and_reset(graph):
    fs, ms, nbytes, S, P = 48000, 10, 120, 96, 20
    rng = np.random.default_rng(23)
    resets = {5: rng.permutation(S)[:40].astype(np.int32), 12: rng.permutation(S)[:20].astype(np.int32)}
    pcm, _ = corpus(fs, ms, nbytes, S + 60, P)
    enc = _encoder(fs, ms, S, nbytes, graph=graph)
    book, got = _run_encoder_schedule(enc, S, _schedule(S, P, rng), pcm, nbytes, resets)
    assert book.n_seq == S + 60
    _check_encoder(got, gpu_encode(fs, ms, pcm, nbytes))


def test_encoder_both_bitstream_paths():
    """Calls below 12 288 rows run the range coder inside the finish kernel, larger ones use the thread-per-frame kernel."""
    fs, ms, nbytes, S = 48000, 10, 120, 13000
    rng = np.random.default_rng(29)
    pcm = make_pcm(S, 4, fs, 480)
    sched = [rng.permutation(S)[:n].astype(np.int32) for n in (12500, 3000, 12288, 13000)]
    enc = _encoder(fs, ms, S, nbytes)
    _, got = _run_encoder_schedule(enc, S, sched, pcm, nbytes)
    _check_encoder(got, gpu_encode(fs, ms, pcm, nbytes))


def test_encoder_gate_against_oracle():
    fs, ms, nbytes, S, P = 32000, 7.5, 70, 96, 30
    rng = np.random.default_rng(31)
    pcm, o_frames = corpus(fs, ms, nbytes, S, P)
    enc = _encoder(fs, ms, S, nbytes)
    book, got = _run_encoder_schedule(enc, S, _schedule(S, P, rng), pcm, nbytes)
    m = 8                                                         # streams that had at least m frames, first m of them
    keep = [s for s in range(S) if book.cnt[s] >= m]
    assert len(keep) >= 48
    g = np.array([[got[(s, k)] for k in range(m)] for s in keep])
    encoder_gate(pcm[keep, :m], o_frames[keep, :m], g, fs, ms)


def test_encoder_rejects_bad_id_lists():
    import torch

    import lc3_codec_b200 as L
    fs, ms, nbytes, S = 48000, 10, 120, 16
    enc = _encoder(fs, ms, S, nbytes)
    lib = L.lib()
    x = torch.zeros((S, 480), dtype=torch.int16, device="cuda:0")
    y = torch.zeros((S, nbytes), dtype=torch.uint8, device="cuda:0")
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(ids, n):
        arr = None if ids is None else np.ascontiguousarray(ids, dtype=np.int32)
        p = None if arr is None else C.c_void_p(arr.ctypes.data)
        return lib.lc3b_encode_frames_subset(enc._h, p, n, C.c_void_p(x.data_ptr()), 480, C.c_void_p(y.data_ptr()),
                                             nbytes, nbytes, stream)

    assert call(None, 1) == 2
    assert call([0], -1) == 2
    assert call(np.arange(S + 1), S + 1) == 2
    assert call([S], 1) == 2 and call([-3], 1) == 2
    assert call([1, 4, 1], 3) == 2
    assert call([], 0) == 0 and call([2, 0], 2) == 0
    assert lib.lc3b_encoder_reset_streams(enc._h, None, 1, stream) == 2
    torch.cuda.synchronize()
