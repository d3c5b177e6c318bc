"""Ragged time-parallel calls (lc3b_decode_stream_frames_subset, lc3b_encode_stream_frames_subset).

Contract: row i of a call equals frame_counts[i] frame-by-frame calls on stream stream_ids[i] - PCM, status and bytes,
and every piece of per-stream state afterwards.  The reference is a "lockstep" handle with one row per stream sequence
driven frame by frame (as in test_stream_subset_gpu.py); exact equality is required.  Every check ends with further
frame-by-frame calls, which catch a state hand-back error the call's own output cannot show.
"""
import ctypes as C

import numpy as np
import pytest

from common import corpus, encoder_gate, gpu_decode, gpu_encode
from tools.corpus import make_pcm

pytestmark = pytest.mark.gpu

COUNTS = (0, 1, 2, 7, 33, 200)
MORE = 10                                                         # frame-by-frame calls after the ragged ones


def _decoder(fs, ms, S, nb, **opts):
    import torch

    import lc3_codec_b200 as L
    sf, fd = L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)
    ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(S, fd, sf, nb), dtype=torch.uint8, device="cuda:0")
    dec = L.Lc3BatchDecoder(S, fd, sf, ws, nb)
    for k, v in opts.items():
        getattr(dec, "set_" + k)(v)
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
        self.seq, self.cnt, self.n_seq = list(range(S)), [0] * S, S

    def take(self, ids, counts):
        """(seq, k) of every unit of a ragged call, rows packed in the caller's order."""
        vk = []
        for s, c in zip(ids, counts):
            vk += [(self.seq[s], self.cnt[s] + f) for f in range(c)]
            self.cnt[s] += int(c)
        return vk

    def reset(self, ids):
        for s in ids:
            self.seq[s], self.cnt[s] = self.n_seq, 0
            self.n_seq += 1


def _ragged_decode(dec, ids, counts, book, frames, lens, got):
    import torch
    vk = book.take(ids, counts)
    V = len(vk)
    fr = np.array([frames[v, k] for v, k in vk], np.uint8).reshape(V, frames.shape[2])
    ln = None if lens is None else torch.from_numpy(np.array([lens[v, k] for v, k in vk], np.int32)).cuda()
    out = torch.full((V * dec.nf,), 12345, dtype=torch.int16, device="cuda:0")
    st = torch.full((V,), 7, dtype=torch.int32, device="cuda:0")
    scratch = torch.empty(dec.multi_subset_scratch_bytes(len(ids), V), dtype=torch.uint8, device="cuda:0")
    dec.decode_stream_frames_subset(16, ids, counts, torch.from_numpy(fr).cuda(), out, scratch, ln, st)
    out, st = out.cpu().numpy().reshape(V, dec.nf), st.cpu().numpy()
    for i, key in enumerate(vk):
        got[key] = (out[i], st[i])


def _full_decode(dec, S, book, frames, lens, got):
    import torch
    vk = book.take(range(S), [1] * S)
    fr = np.array([frames[v, k] for v, k in vk], np.uint8)
    ln = None if lens is None else torch.from_numpy(np.array([lens[v, k] for v, k in vk], np.int32)).cuda()
    out = torch.zeros((S, dec.nf), dtype=torch.int16, device="cuda:0")
    st = torch.zeros(S, dtype=torch.int32, device="cuda:0")
    dec.decode_frames(16, torch.from_numpy(fr).cuda(), out, ln, status_out=st)
    for i, key in enumerate(vk):
        got[key] = (out[i].cpu().numpy(), int(st[i]))


def _check_decoder(book, got, ref, spectrum_now, S):
    r_pcm, _tr, _x, r_sp, r_status = ref
    for (v, k), (pcm, st) in got.items():
        assert np.array_equal(pcm, r_pcm[v, k]), f"PCM of sequence {v} frame {k} differs from the lockstep handle"
        assert st == r_status[v, k], f"status of sequence {v} frame {k}"
    if spectrum_now is None:
        return
    for s in range(S):
        v, n = book.seq[s], book.cnt[s]
        want = r_sp[v, n - 1] if n else np.zeros_like(r_sp[0, 0])
        assert np.array_equal(spectrum_now[s].view(np.uint32), want.view(np.uint32)), f"spectrum of stream {s}"


def _rows(S, rng, choices=COUNTS):
    ids = rng.permutation(S).astype(np.int32)
    counts = rng.choice(choices, S).astype(np.int32)
    counts[:len(choices)] = choices                               # every count at least once
    return ids, counts


DEC_CASES = [(48000, 10, 150, False), (16000, 7.5, 30, False), (24000, 10, 40, True)]


@pytest.mark.parametrize("fs,ms,nbytes,lossy", DEC_CASES)
def test_decoder_ragged_equals_lockstep(fs, ms, nbytes, lossy):
    """16 kHz / 7.5 ms / 30 B runs the post filter with its 3-block ring; the lossy case has lost and bit-flipped frames,
    a loss at a row's first and at its last frame and a row that is entirely lost."""
    S = 24
    rng = np.random.default_rng(41)
    ids, counts = _rows(S, rng)
    ids2, counts2 = _rows(S, rng, (0, 1, 2, 7))
    P = int(counts.max() + counts2.max()) + MORE
    _, frames = corpus(fs, ms, nbytes, S, P)
    frames, lens = frames.copy(), None
    if lossy:
        lens = np.full((S, P), nbytes, np.int32)
        lens[rng.random((S, P)) < 0.08] = 0
        flip = rng.random((S, P)) < 0.08
        frames[flip, 3] ^= 0x5A
        by_count = {int(c): int(s) for s, c in zip(ids, counts)}
        lens[by_count[33], 0] = 0                                 # first frame of a row
        lens[by_count[200], 199] = 0                              # last frame of a row
        lens[by_count[7], :7] = 0                                 # a row that is entirely lost
    dec = _decoder(fs, ms, S, nbytes)
    book, got = Book(S), {}
    _ragged_decode(dec, ids, counts, book, frames, lens, got)
    ref = gpu_decode(fs, ms, frames, lens)
    _check_decoder(book, got, ref, dec.spectrum().cpu().numpy(), S)
    _ragged_decode(dec, ids2, counts2, book, frames, lens, got)
    _check_decoder(book, got, ref, dec.spectrum().cpu().numpy(), S)
    for _ in range(MORE):
        _full_decode(dec, S, book, frames, lens, got)
    _check_decoder(book, got, ref, dec.spectrum().cpu().numpy(), S)
    if lossy:
        assert any(st == 1 for _, st in got.values())


def test_decoder_equal_counts_identity_ids_equal_dense_call():
    import torch
    fs, ms, nbytes, S, F = 16000, 7.5, 30, 40, 12
    _, frames = corpus(fs, ms, nbytes, S, F)
    a, b = _decoder(fs, ms, S, nbytes), _decoder(fs, ms, S, nbytes)
    fr = torch.from_numpy(np.ascontiguousarray(frames)).cuda()
    out_a = torch.zeros((S, F * a.nf), dtype=torch.int16, device="cuda:0")
    out_b = torch.ones(S * F * b.nf, dtype=torch.int16, device="cuda:0")
    st_a = torch.zeros((S, F), dtype=torch.int32, device="cuda:0")
    st_b = torch.ones(S * F, dtype=torch.int32, device="cuda:0")
    a.decode_stream_frames(16, fr, out_a, torch.empty(a.multi_scratch_bytes(F), dtype=torch.uint8, device="cuda:0"),
                           status_out=st_a)
    b.decode_stream_frames_subset(16, np.arange(S), np.full(S, F), fr.reshape(S * F, nbytes), out_b,
                                  torch.empty(b.multi_subset_scratch_bytes(S, S * F), dtype=torch.uint8, device="cuda:0"),
                                  status_out=st_b)
    assert torch.equal(out_a.reshape(-1), out_b) and torch.equal(st_a.reshape(-1), st_b)
    assert torch.equal(a.spectrum(), b.spectrum())


def test_decoder_ragged_interleaved_with_every_other_call_and_resets():
    import torch
    fs, ms, nbytes, S = 16000, 7.5, 30, 48
    rng = np.random.default_rng(43)
    _, frames = corpus(fs, ms, nbytes, S + 40, 80)
    dec = _decoder(fs, ms, S, nbytes)
    book, got = Book(S), {}
    for step in range(4):
        ids, counts = _rows(S, rng, (0, 1, 2, 7))
        _ragged_decode(dec, ids, counts, book, frames, None, got)
        sub = rng.permutation(S)[:int(rng.integers(1, S))].astype(np.int32)   # a subset call
        vk = book.take(sub, [1] * len(sub))
        out = torch.zeros((len(sub), dec.nf), dtype=torch.int16, device="cuda:0")
        st = torch.zeros(len(sub), dtype=torch.int32, device="cuda:0")
        dec.decode_frames_subset(16, sub, torch.from_numpy(np.array([frames[v, k] for v, k in vk], np.uint8)).cuda(), out,
                                 status_out=st)
        for i, key in enumerate(vk):
            got[key] = (out[i].cpu().numpy(), int(st[i]))
        if step == 1:                                             # a dense time-parallel call
            F = 3
            vk = book.take(range(S), [F] * S)
            blk = np.array([frames[v, k] for v, k in vk], np.uint8).reshape(S, F, nbytes)
            out = torch.zeros((S, F * dec.nf), dtype=torch.int16, device="cuda:0")
            st = torch.zeros((S, F), dtype=torch.int32, device="cuda:0")
            dec.decode_stream_frames(16, torch.from_numpy(blk).cuda(), out,
                                     torch.empty(dec.multi_scratch_bytes(F), dtype=torch.uint8, device="cuda:0"), status_out=st)
            out, st = out.cpu().numpy().reshape(S * F, dec.nf), st.cpu().numpy().reshape(-1)
            for i, key in enumerate(vk):
                got[key] = (out[i], st[i])
        if step == 2:
            r = rng.permutation(S)[:20].astype(np.int32)
            dec.reset_streams(r)
            book.reset(r)
        _full_decode(dec, S, book, frames, None, got)
    assert book.n_seq == S + 20
    _check_decoder(book, got, gpu_decode(fs, ms, frames), dec.spectrum().cpu().numpy(), S)


@pytest.mark.parametrize("split,dequant_mode", [(1, 1), (4, 2), (1, 2), (4, 0)])
def test_decoder_large_ragged_call(split, dequant_mode):
    """>= 65 536 units: the entropy stage of a split call runs as four sub-batches.  Frames from the engine's encoder."""
    fs, ms, nbytes, S = 16000, 7.5, 30, 640
    rng = np.random.default_rng(47)
    counts = rng.integers(0, 231, S).astype(np.int32)
    counts[:3] = (0, 1, 230)
    ids = rng.permutation(S).astype(np.int32)
    assert counts.sum() >= 65536
    P = 230 + MORE
    frames = gpu_encode(fs, ms, make_pcm(S, P, fs, 120), nbytes)
    lens = np.full((S, P), nbytes, np.int32)
    lens[rng.random((S, P)) < 0.03] = 0
    dec = _decoder(fs, ms, S, nbytes, split=split, dequant_mode=dequant_mode)
    book, got = Book(S), {}
    _ragged_decode(dec, ids, counts, book, frames, lens, got)
    for _ in range(MORE):
        _full_decode(dec, S, book, frames, lens, got)
    _check_decoder(book, got, gpu_decode(fs, ms, frames, lens, trace=False), None, S)


def _dec_error_setup():
    import torch
    fs, ms, nbytes, S = 48000, 10, 150, 16
    _, frames = corpus(fs, ms, nbytes, S, 4)
    dec = _decoder(fs, ms, S, nbytes)
    V = 8
    fr = torch.from_numpy(np.ascontiguousarray(frames[:, :2].reshape(-1, nbytes)[:V])).cuda()
    out = torch.full((V * dec.nf,), 777, dtype=torch.int16, device="cuda:0")
    st = torch.full((V,), 9, dtype=torch.int32, device="cuda:0")
    return dec, frames, fr, out, st, V


def test_decoder_rejects_bad_calls_and_enqueues_nothing():
    import torch

    import lc3_codec_b200 as L
    dec, frames, fr, out, st, V = _dec_error_setup()
    lib = L.lib()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    need = dec.multi_subset_scratch_bytes(3, V)
    big = torch.empty(need + 512, dtype=torch.uint8, device="cuda:0")

    def call(ids, counts, scratch_off=0, scratch_bytes=need, bits=16):
        a = np.ascontiguousarray(ids, dtype=np.int32)
        c = np.ascontiguousarray(counts, dtype=np.int32)
        return lib.lc3b_decode_stream_frames_subset(
            dec._h, bits, C.c_void_p(a.ctypes.data), C.c_void_p(c.ctypes.data), a.size, C.c_void_p(fr.data_ptr()), None,
            150, 150, C.c_void_p(out.data_ptr()), C.c_void_p(st.data_ptr()), C.c_void_p(big.data_ptr() + scratch_off),
            scratch_bytes, stream)

    assert call([0, 16, 2], [3, 3, 2]) == 2                       # out of range
    assert call([0, -1, 2], [3, 3, 2]) == 2
    assert call([5, 1, 5], [3, 3, 2]) == 2                        # listed twice
    assert call([5, 1, 2], [3, -1, 6]) == 2                       # negative count
    assert call([5, 1], [0x7fffffff // 512, 1]) == 2              # total over the unit limit
    assert call([5, 1, 2], [3, 3, 2], scratch_bytes=need - 1) == 4
    assert call([5, 1, 2], [3, 3, 2], scratch_off=4) == 4         # misaligned
    assert call([5, 1, 2], [3, 3, 2], bits=8) == 1
    assert call([], []) == 0 and call([5, 1, 2], [0, 0, 0]) == 0   # nothing to do
    n = C.c_size_t(0)
    assert lib.lc3b_decoder_multi_subset_scratch_bytes(dec._h, 17, 1, C.byref(n)) == 2
    assert lib.lc3b_decoder_multi_subset_scratch_bytes(dec._h, 1, -1, C.byref(n)) == 2
    assert lib.lc3b_decoder_multi_subset_scratch_bytes(dec._h, 1, 0x7fffffff // 512 + 1, C.byref(n)) == 2
    torch.cuda.synchronize()
    assert (out.cpu().numpy() == 777).all() and (st.cpu().numpy() == 9).all()
    # no stream moved on: a frame-by-frame call continues from frame 0
    S = frames.shape[0]
    out2 = torch.zeros((S, dec.nf), dtype=torch.int16, device="cuda:0")
    dec.decode_frames(16, torch.from_numpy(np.ascontiguousarray(frames[:, 0])).cuda(), out2)
    assert np.array_equal(out2.cpu().numpy(), gpu_decode(48000, 10, frames[:, :1], trace=False)[0][:, 0])


# ---------------------------------------------------------------------------------------------------------- encoder
def _ragged_encode(enc, ids, counts, book, pcm, nbytes, got):
    import torch
    vk = book.take(ids, counts)
    V = len(vk)
    x = np.array([pcm[v, k] for v, k in vk], np.int16).reshape(V * pcm.shape[2])
    out = torch.zeros((V, nbytes), dtype=torch.uint8, device="cuda:0")
    scratch = torch.empty(enc.multi_subset_scratch_bytes(len(ids), V), dtype=torch.uint8, device="cuda:0")
    enc.encode_stream_frames_subset(ids, counts, torch.from_numpy(x).cuda(), out, scratch)
    out = out.cpu().numpy()
    for i, key in enumerate(vk):
        got[key] = out[i]


def _full_encode(enc, S, book, pcm, nbytes, got):
    import torch
    vk = book.take(range(S), [1] * S)
    out = torch.zeros((S, nbytes), dtype=torch.uint8, device="cuda:0")
    enc.encode_frames(torch.from_numpy(np.array([pcm[v, k] for v, k in vk], np.int16)).cuda(), out)
    out = out.cpu().numpy()
    for i, key in enumerate(vk):
        got[key] = out[i]


def _check_encoder(got, ref):
    for (v, k), b in got.items():
        assert np.array_equal(b, ref[v, k]), f"bytes of sequence {v} frame {k} differ from the lockstep handle"


# counts that differ inside one CTA of the LTPF walk (4 warps) and of the quantiser walk (8 warps), in caller order
MIX = [1, 1, 50, 3, 0, 120, 2, 7, 33, 0, 1, 64, 5, 5, 90, 2, 0, 11, 1, 40, 3, 70, 0, 9, 2, 1, 18, 6, 0, 100, 4, 1]


@pytest.mark.parametrize("fs,ms,nbytes,graph", [(16000, 7.5, 30, False), (24000, 10, 40, True), (48000, 10, 120, False),
                                                 (32000, 7.5, 70, True)])
def test_encoder_ragged_equals_lockstep(fs, ms, nbytes, graph):
    S = len(MIX)
    rng = np.random.default_rng(53)
    ids = rng.permutation(S).astype(np.int32)
    counts = np.array(MIX, np.int32)
    ids2, counts2 = rng.permutation(S).astype(np.int32), rng.choice([0, 1, 2, 7], S).astype(np.int32)
    P = int(counts.max() + counts2.max()) + MORE
    enc = _encoder(fs, ms, S, nbytes, graph=graph)
    pcm = make_pcm(S, P, fs, enc.nf)
    book, got = Book(S), {}
    _ragged_encode(enc, ids, counts, book, pcm, nbytes, got)
    _ragged_encode(enc, ids2, counts2, book, pcm, nbytes, got)
    for _ in range(MORE):
        _full_encode(enc, S, book, pcm, nbytes, got)
    _check_encoder(got, gpu_encode(fs, ms, pcm, nbytes))


def test_encoder_equal_counts_identity_ids_equal_dense_call():
    import torch
    fs, ms, nbytes, S, F = 48000, 10, 120, 24, 9
    pcm = make_pcm(S, F + 1, fs, 480)
    a, b = _encoder(fs, ms, S, nbytes), _encoder(fs, ms, S, nbytes)
    x = torch.from_numpy(np.ascontiguousarray(pcm[:, :F].reshape(S, F * 480))).cuda()
    ya = torch.zeros((S, F, nbytes), dtype=torch.uint8, device="cuda:0")
    yb = torch.ones((S * F, nbytes), dtype=torch.uint8, device="cuda:0")
    a.encode_stream_frames(x, ya, torch.empty(a.multi_scratch_bytes(F), dtype=torch.uint8, device="cuda:0"))
    b.encode_stream_frames_subset(np.arange(S), np.full(S, F), x.reshape(-1), yb,
                                  torch.empty(b.multi_subset_scratch_bytes(S, S * F), dtype=torch.uint8, device="cuda:0"))
    assert torch.equal(ya.reshape(S * F, nbytes), yb)
    za, zb = (torch.zeros((S, nbytes), dtype=torch.uint8, device="cuda:0") for _ in range(2))
    nxt = torch.from_numpy(pcm[:, F].copy()).cuda()
    a.encode_frames(nxt, za)
    b.encode_frames(nxt, zb)
    assert torch.equal(za, zb)


def test_encoder_ragged_gate_against_oracle_and_resets():
    fs, ms, nbytes, S = 32000, 7.5, 70, 32
    rng = np.random.default_rng(59)
    pcm, o_frames = corpus(fs, ms, nbytes, S + 16, 40)
    enc = _encoder(fs, ms, S, nbytes)
    book, got = Book(S), {}
    _ragged_encode(enc, rng.permutation(S).astype(np.int32), np.array(MIX, np.int32) % 17, book, pcm, nbytes, got)
    r = rng.permutation(S)[:16].astype(np.int32)
    enc.reset_streams(r)
    book.reset(r)
    _ragged_encode(enc, rng.permutation(S).astype(np.int32), rng.choice([0, 1, 2, 7], S).astype(np.int32), book, pcm, nbytes, got)
    for _ in range(MORE):
        _full_encode(enc, S, book, pcm, nbytes, got)
    _check_encoder(got, gpu_encode(fs, ms, pcm, nbytes))
    m = 10
    keep = [v for v in range(S + 16) if all((v, k) in got for k in range(m))]
    assert len(keep) >= 24
    encoder_gate(pcm[keep, :m], o_frames[keep, :m], np.array([[got[(v, k)] for k in range(m)] for v in keep]), fs, ms)


def test_encoder_rejects_bad_calls_and_enqueues_nothing():
    import torch

    import lc3_codec_b200 as L
    fs, ms, nbytes, S, V = 48000, 10, 120, 16, 8
    enc = _encoder(fs, ms, S, nbytes)
    lib = L.lib()
    pcm = make_pcm(S, 2, fs, 480)
    x = torch.zeros(V * 480, dtype=torch.int16, device="cuda:0")
    y = torch.full((V, nbytes), 0xAB, dtype=torch.uint8, device="cuda:0")
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    need = enc.multi_subset_scratch_bytes(3, V)
    big = torch.empty(need + 512, dtype=torch.uint8, device="cuda:0")

    def call(ids, counts, scratch_off=0, scratch_bytes=need):
        a = np.ascontiguousarray(ids, dtype=np.int32)
        c = np.ascontiguousarray(counts, dtype=np.int32)
        return lib.lc3b_encode_stream_frames_subset(
            enc._h, C.c_void_p(a.ctypes.data), C.c_void_p(c.ctypes.data), a.size, C.c_void_p(x.data_ptr()),
            C.c_void_p(y.data_ptr()), nbytes, nbytes, C.c_void_p(big.data_ptr() + scratch_off), scratch_bytes, stream)

    assert call([0, 16, 2], [3, 3, 2]) == 2
    assert call([0, -2, 2], [3, 3, 2]) == 2
    assert call([4, 4], [3, 3]) == 2
    assert call([5, 1, 2], [3, 3, -2]) == 2
    assert call([5, 1], [0x7fffffff, 1]) == 2                     # total beyond an int
    assert call([5, 1, 2], [3, 3, 2], scratch_bytes=need - 1) == 4
    assert call([5, 1, 2], [3, 3, 2], scratch_off=8) == 4
    assert call([], []) == 0 and call([3], [0]) == 0
    n = C.c_size_t(0)
    assert lib.lc3b_encoder_multi_subset_scratch_bytes(enc._h, 17, 1, C.byref(n)) == 2
    assert lib.lc3b_encoder_multi_subset_scratch_bytes(enc._h, 1, 2**31, C.byref(n)) == 2
    torch.cuda.synchronize()
    assert (y.cpu().numpy() == 0xAB).all()
    ya = torch.zeros((S, nbytes), dtype=torch.uint8, device="cuda:0")
    enc.encode_frames(torch.from_numpy(pcm[:, 0].copy()).cuda(), ya)   # no stream moved on
    assert np.array_equal(ya.cpu().numpy(), gpu_encode(fs, ms, pcm[:, :1], nbytes)[:, 0])
