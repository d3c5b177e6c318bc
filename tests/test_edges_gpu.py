"""GPU parity at the codec's edges: every frame length from 1 to 400 bytes, frame lengths on either side of each integer
rate decision the reference makes, and the edge material of tools/edge_corpus.py (silence, full scale, steps, pulse
trains, ...), against the oracle.

The rate boundaries come from the reference's formulas (tools/edge_corpus.rate_boundaries), not from the engine.  The
bars are the suite's: encoder bytes identical on every frame; decoder traces and integer spectra bit exact, the shaped
spectrum bit exact on decoded frames, PCM bit exact against the oracle run with the engine's inverse MDCT and within
+-1 LSB against the oracle run with the reference's (a difference bounded by the float64 DCT-IV test of
tests/test_engine_transform_cpu.py).
"""
import ctypes as C
import functools

import numpy as np
import pytest

from common import ALL_CONFIGS, assert_parity, assert_pcm_matches_oracle, gpu_decode, gpu_encode
from oracle import pyoracle as O
from tools import edge_corpus as E

pytestmark = pytest.mark.gpu

ENC_CONFIGS = [k for k in ALL_CONFIGS if k[0] != 8000]
N_CLS = len(E.CLASSES)
LENGTHS = np.arange(E.MIN_NBYTES, E.MAX_NBYTES + 1)


def _fs_ind(fs, ms):
    return O.config(fs, ms)["fs_ind"]


def _enc_material(fs, ms, n_frames, n_var=2, n_corpus=4):
    """Every edge class in n_var variants, then n_corpus streams of the synthetic corpus."""
    nf = O.config(fs, ms)["nf"]
    from tools.corpus import make_pcm
    return np.concatenate([E.make_edge_pcm(N_CLS * n_var, n_frames, fs, ms),
                           make_pcm(n_corpus, n_frames, fs, nf, first_stream=1)])


def _encoder(fs, ms, S, nb):
    import torch

    import lc3_codec_b200 as L
    sf, fd = L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)
    ws = torch.empty(L.Lc3BatchEncoder.calc_working_buffer_lengths(S, fd, sf, nb), dtype=torch.uint8, device="cuda:0")
    return L.Lc3BatchEncoder(S, fd, sf, ws, nb)


def _encode_multi(fs, ms, pcm, nbytes):
    """pcm [S, F, nf] -> bytes [S, F, nbytes] through one lc3b_encode_stream_frames call of a fresh handle."""
    import torch
    S, F, nf = pcm.shape
    enc = _encoder(fs, ms, S, nbytes)
    scratch = torch.empty(enc.multi_scratch_bytes(F), dtype=torch.uint8, device="cuda:0")
    out = torch.zeros((S, F, nbytes), dtype=torch.uint8, device="cuda:0")
    enc.encode_stream_frames(torch.from_numpy(np.ascontiguousarray(pcm.reshape(S, F * nf))).cuda(), out, scratch)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def _decoder(fs, ms, S, max_nbytes=E.MAX_NBYTES):
    import torch

    import lc3_codec_b200 as L
    sf, fd = L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)
    ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(S, fd, sf, max_nbytes), dtype=torch.uint8, device="cuda:0")
    return L.Lc3BatchDecoder(S, fd, sf, ws, max_nbytes)


def _decode_multi(fs, ms, frames, lens, min_nbytes=0):
    """frames [S, F, nb] -> (pcm [S, F, nf], status [S, F]) through one lc3b_decode_stream_frames call."""
    import torch
    S, F, nb = frames.shape
    dec = _decoder(fs, ms, S, nb)
    if min_nbytes:
        dec.set_min_nbytes(min_nbytes)
    scratch = torch.empty(dec.multi_scratch_bytes(F), dtype=torch.uint8, device="cuda:0")
    out = torch.zeros((S, F * dec.nf), dtype=torch.int16, device="cuda:0")
    st = torch.zeros((S, F), dtype=torch.int32, device="cuda:0")
    ln = torch.from_numpy(np.ascontiguousarray(lens.astype(np.int32))).cuda()
    dec.decode_stream_frames(16, torch.from_numpy(np.ascontiguousarray(frames)).cuda(), out, scratch, ln, st)
    torch.cuda.synchronize()
    return out.cpu().numpy().reshape(S, F, dec.nf), st.cpu().numpy()


def _assert_bytes_equal(o, g, what):
    bad = np.argwhere((o != g).any(-1))
    assert bad.size == 0, f"{what}: {len(bad)} frames differ, first (stream, frame) {bad[:6].tolist()}"


# ------------------------------------------------------------------------------------------------------------- encoder
@pytest.mark.parametrize("fs,ms", ENC_CONFIGS)
def test_encoder_at_every_rate_boundary(fs, ms):
    """Edge material and corpus streams at b - 1, b, b + 1 of every boundary and at 20, 21, 399, 400 B: one
    lc3b_encode_stream_frames call per length, bytes identical to the oracle on every frame; the first length also
    frame by frame through lc3b_encode_frames."""
    F = 6
    pcm = _enc_material(fs, ms, F)
    lengths = E.boundary_lengths(_fs_ind(fs, ms), fs, ms)
    for i, nb in enumerate(lengths):
        o = O.encode_streams(pcm, fs, ms, nb)
        _assert_bytes_equal(o, _encode_multi(fs, ms, pcm, nb), (fs, ms, nb, "encode_stream_frames"))
        if i == 0:
            _assert_bytes_equal(o, gpu_encode(fs, ms, pcm, nb), (fs, ms, nb, "encode_frames"))


@pytest.mark.parametrize("fs,ms", ENC_CONFIGS)
def test_encoder_sparse_sweep_of_every_length(fs, ms):
    """Every length from 20 to 400 B: two streams of four frames, the edge class rotating with the length."""
    F = 4
    for nb in LENGTHS:
        pcm = E.make_edge_pcm(2, F, fs, ms, first_stream=2 * int(nb))
        _assert_bytes_equal(O.encode_streams(pcm, fs, ms, int(nb)), _encode_multi(fs, ms, pcm, int(nb)), (fs, ms, nb))


@pytest.mark.parametrize("fs,ms", [(48000, 10), (16000, 7.5)])
@pytest.mark.parametrize("nbytes", [20, 100, 400])
def test_encoder_stage_parity_on_edge_material(fs, ms, nbytes):
    """lc3b_encoder_debug_read against the oracle's stages chained by hand (as test_encoder_gpu.py does on the corpus):
    band energies, the attack / LTPF decisions, the quantiser's input and the quantised spectrum, bit for bit."""
    lib = O.lib()
    sf, fd = O.SF[fs], O.FD[ms]
    cfg = O.config(fs, ms)
    nf, ne, fs_ind = cfg["nf"], cfg["ne"], cfg["fs_ind"]
    F = 5
    pcm = E.make_edge_pcm(N_CLS, F, fs, ms)
    _, dbg = gpu_encode(fs, ms, pcm, nbytes, debug=True)
    nbits = nbytes * 8
    attacks = 0
    for s_ in range(pcm.shape[0]):
        mdct, att, ltpf = (C.c_void_p(getattr(lib, f"lc3o_{n}_new")(sf, fd)) for n in ("encmdct", "attack", "encltpf"))
        quant = C.c_void_p(lib.lc3o_quant_new(ne, fs_ind))
        for f in range(F):
            x16 = np.ascontiguousarray(pcm[s_, f])
            spec, eb = np.zeros(nf, np.float32), np.zeros(64, np.float32)
            near_nyquist = lib.lc3o_encmdct_run(mdct, O.p(x16), O.p(spec), O.p(eb))
            attack = lib.lc3o_attack_run(att, O.p(x16), nbytes)
            attacks += attack
            lt = np.zeros(4, np.int32)
            lib.lc3o_encltpf_run(ltpf, O.p(x16), near_nyquist, nbits, O.p(lt))
            bw = np.zeros(2, np.int32)
            lib.lc3o_bandwidth_detect(sf, fd, O.p(eb), O.p(bw))
            sns = np.zeros(7, np.int64)
            lib.lc3o_sns_encode(sf, fd, O.p(spec), O.p(eb), attack, O.p(sns))
            ti, rq = np.zeros(21, np.int32), np.zeros(16, np.float32)
            lib.lc3o_tns_encode(sf, fd, O.p(spec), int(bw[0]), nbits, near_nyquist, O.p(ti), O.p(rq))
            xq, qi, gg = np.zeros(ne, np.int16), np.zeros(7, np.int32), C.c_float(0)
            lib.lc3o_quant_run(quant, O.p(spec), O.p(xq), nbits, int(bw[1]), int(ti[0]), int(lt[3]), O.p(qi), C.byref(gg))
            g_xf, g_eb, g_hand, g_xq = (a[s_] for a in dbg[f])
            where = (fs, ms, nbytes, E.edge_class(s_), f)
            assert np.array_equal(g_eb.view(np.uint32), eb.view(np.uint32)), where
            assert g_hand[:6].tolist() == [near_nyquist, attack, int(lt[0]), int(lt[1]), int(lt[2]), int(lt[3])], where
            assert np.array_equal(g_xf.view(np.uint32), spec[:ne].view(np.uint32)), where
            assert np.array_equal(g_xq, xq), where
        lib.lc3o_encmdct_free(mdct)
        lib.lc3o_attack_free(att)
        lib.lc3o_encltpf_free(ltpf)
        lib.lc3o_quant_free(quant)
    if fs == 48000 and nbytes >= 100:
        assert attacks > 0


# ------------------------------------------------------------------------------------------------------------- decoder
@functools.lru_cache(maxsize=2)
def _every_length_batch(fs, ms, F=4):
    """381 streams, stream i carrying oracle-encoded frames of 20 + i bytes of edge stream i: (frames [381, F, 400], lens)."""
    pcm = E.make_edge_pcm(len(LENGTHS), F, fs, ms)
    frames = np.zeros((len(LENGTHS), F, E.MAX_NBYTES), np.uint8)
    for i, nb in enumerate(LENGTHS):
        frames[i, :, :nb] = O.encode_streams(pcm[i:i + 1], fs, ms, int(nb))[0]
    lens = np.repeat(LENGTHS[:, None], F, 1).astype(np.int32)
    return frames, lens


@pytest.mark.parametrize("fs,ms", ALL_CONFIGS)
def test_decoder_every_length_in_one_batch(fs, ms):
    """Every length from 20 to 400 B side by side through frame_nbytes: both dequantisation kernels, four sub-batches,
    and the time-parallel call bit-identical to the frame-by-frame one, status included."""
    frames, lens = _every_length_batch(fs, ms)
    for mode in (1, 2):
        assert_parity(fs, ms, frames, lens, dequant_mode=mode)
    assert_parity(fs, ms, frames, lens, split=4)
    g_pcm, _, _, _, g_st = gpu_decode(fs, ms, frames, lens, trace=False)
    m_pcm, m_st = _decode_multi(fs, ms, frames, lens)
    assert np.array_equal(m_pcm, g_pcm) and np.array_equal(m_st, g_st)
    # the reference's own decoder rejects a few of its encoder's frames (NegativeResidualNumBits: full-scale noise and
    # steps at 24 and 41 B at 44.1 / 48 kHz / 10 ms, noise at 32 B at 16 kHz / 7.5 ms); assert_parity holds the engine to
    # the same status on every frame, here only that such frames stay rare
    assert (g_st == 1).mean() < 0.01


def test_mixed_decoder_every_length_every_config():
    """One Lc3MixedBatchDecoder call over the 12 x 381 rows of the every-length batches equals each configuration's
    own handle."""
    import torch

    import lc3_codec_b200 as L
    F = 2
    batches = {k: _every_length_batch(*k)[0][:, :F] for k in ALL_CONFIGS}
    cfgs, rows, lens = [], [], []
    for k in ALL_CONFIGS:
        cfgs += [k] * len(LENGTHS)
        rows.append(batches[k])
        lens.append(np.repeat(LENGTHS[:, None], F, 1))
    frames, lens = np.concatenate(rows), np.concatenate(lens).astype(np.int32)
    dec = L.Lc3MixedBatchDecoder([(L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)) for fs, ms in cfgs],
                                 max_nbytes=E.MAX_NBYTES, device="cuda:0")
    order = np.array(dec.order)                                          # row -> stream
    got = np.zeros((len(cfgs), F, dec.max_nf), np.int16)
    for f in range(F):
        y = torch.zeros((len(cfgs), dec.max_nf), dtype=torch.int16, device="cuda:0")
        dec.decode_frames(16, torch.from_numpy(np.ascontiguousarray(frames[order, f])).cuda(),
                          torch.from_numpy(np.ascontiguousarray(lens[order, f])).cuda(), y)
        torch.cuda.synchronize()
        got[order, f] = y.cpu().numpy()
    r = 0
    for k in ALL_CONFIGS:
        nf = O.config(*k)["nf"]
        single = gpu_decode(*k, batches[k], lens[r:r + len(LENGTHS)], trace=False)[0]
        assert np.array_equal(got[r:r + len(LENGTHS), :, :nf], single), k
        r += len(LENGTHS)


@functools.lru_cache(maxsize=2)
def _pitched(fs, ms, S, F):
    """Pulse trains at lag 36 and 228 and the lag jump, plus speech-like corpus streams: material the LTPF takes."""
    nf = O.config(fs, ms)["nf"]
    from tools.corpus import make_pcm
    pulses = E.make_edge_streams(E.streams_of("pulses", 4)[1:], F, fs, ms)
    speech = make_pcm(3 * (S - 3), F, fs, nf)[2::3]                      # corpus class 2: speech-like
    return np.concatenate([pulses, speech])


@pytest.mark.parametrize("fs,ms", ALL_CONFIGS)
def test_lengths_alternating_across_each_post_filter_gain_row(fs, ms):
    """Frame f is the oracle's frame f of the same PCM at b - 1 (f even) or b (f odd), for every gain row b of the
    decoder's post filter and its end: the gain changes from frame to frame with the pitch unchanged.  Frame by frame
    and time-parallel."""
    S, F = 12, 12
    pcm = _pitched(fs, ms, S, F)
    fs_ind = _fs_ind(fs, ms)
    rb = E.rate_boundaries(fs_ind, fs, ms)
    active = 0
    for b in rb["ltpf_rows"] + rb["ltpf_gain"]:
        if b - 1 < E.MIN_NBYTES:
            continue
        lo, hi = O.encode_streams(pcm, fs, ms, b - 1), O.encode_streams(pcm, fs, ms, b)
        lens = np.where(np.arange(F)[None, :] % 2 == 0, b - 1, b).repeat(S, 0).astype(np.int32)
        frames = np.zeros((S, F, b), np.uint8)
        frames[:, 0::2, :b - 1] = lo[:, 0::2]
        frames[:, 1::2] = hi[:, 1::2]
        stats = assert_parity(fs, ms, frames, lens)
        active += stats["ltpf_active"]
        m_pcm, _ = _decode_multi(fs, ms, frames, lens)
        assert_pcm_matches_oracle(m_pcm, fs, ms, frames, lens, (fs, ms, b, "decode_stream_frames"))
        assert np.array_equal(m_pcm, gpu_decode(fs, ms, frames, lens, trace=False)[0]), (fs, ms, b)
    assert active > 0


@pytest.mark.parametrize("fs,ms", ALL_CONFIGS)
def test_garbage_at_every_length(fs, ms):
    """Random bytes at every length from 1 to 400 B, the lengths below 20 B that the reader rejects included, plus
    extra streams at the post filter's gain rows (where random side information often leaves the filter active): trace
    parity, and the time-parallel call equals the frame-by-frame one."""
    F = 6
    rb = E.rate_boundaries(_fs_ind(fs, ms), fs, ms)
    rows = [x for b in rb["ltpf_rows"] + rb["ltpf_gain"] for x in (b - 1, b) for _ in range(24)]
    ln = np.concatenate([np.arange(1, E.MAX_NBYTES + 1), rows])
    seed = 0x6A5B + 131 * O.SF[fs] + 7 * O.FD[ms]
    frames = np.random.default_rng(seed).integers(0, 256, (len(ln), F, E.MAX_NBYTES), dtype=np.uint8)
    lens = np.repeat(ln[:, None], F, 1).astype(np.int32)
    for s, n in enumerate(ln):
        frames[s, :, n:] = 0
    stats = assert_parity(fs, ms, frames, lens)
    assert 0.0 < stats["concealed"] < 1.0
    g_pcm = gpu_decode(fs, ms, frames, lens, trace=False)[0]
    m_pcm, _ = _decode_multi(fs, ms, frames, lens)
    assert np.array_equal(m_pcm, g_pcm)


@pytest.mark.parametrize("fs,ms", ALL_CONFIGS)
def test_min_nbytes_promise_at_every_config(fs, ms):
    """T, the reference's first length at which the post filter is impossible: with the promise T, frames of T..400 B
    decode bit-identically to a handle without it and to the oracle; with the promise T - 1, LTPF-active frames of
    T - 1 bytes still match the oracle; frames shorter than the promise are concealed."""
    T = E.ltpf_impossible_from(_fs_ind(fs, ms), ms)
    F = 8
    ln = np.arange(T, E.MAX_NBYTES + 1)
    pcm_all = _pitched(fs, ms, 12, F)
    frames = np.zeros((len(ln), F, E.MAX_NBYTES), np.uint8)
    for i, nb in enumerate(ln):
        frames[i, :, :nb] = O.encode_streams(pcm_all[i % 12:i % 12 + 1], fs, ms, int(nb))[0]
    lens = np.repeat(ln[:, None], F, 1).astype(np.int32)
    assert_parity(fs, ms, frames, lens, min_nbytes=T)
    with_promise = gpu_decode(fs, ms, frames, lens, trace=False, min_nbytes=T)[0]
    assert np.array_equal(with_promise, gpu_decode(fs, ms, frames, lens, trace=False)[0])
    assert np.array_equal(_decode_multi(fs, ms, frames, lens, min_nbytes=T)[0], with_promise)
    # one byte short of T: the filter can act, the handle must keep its history
    below = np.zeros((pcm_all.shape[0], F, E.MAX_NBYTES), np.uint8)
    below[:, :, :T - 1] = O.encode_streams(pcm_all, fs, ms, T - 1)
    lens_b = np.full(below.shape[:2], T - 1, np.int32)
    stats = assert_parity(fs, ms, below, lens_b, min_nbytes=T - 1)
    assert stats["ltpf_active"] > 0
    # shorter than the promise: lost frames, concealed as the oracle conceals an empty frame
    short = np.zeros_like(below)
    short[:, :, :T - 2] = O.encode_streams(pcm_all, fs, ms, T - 2)
    g_pcm, _, _, _, g_st = gpu_decode(fs, ms, short, np.full(short.shape[:2], T - 2, np.int32), trace=False,
                                      min_nbytes=T - 1)
    assert (g_st == 1).all()                                             # all concealed
    assert_pcm_matches_oracle(g_pcm, fs, ms, short, np.zeros(short.shape[:2], np.int32), (fs, ms, "short"))


@pytest.mark.parametrize("fs,ms", ALL_CONFIGS)
def test_edge_material_through_the_decoder(fs, ms):
    """The oracle's bitstreams of the edge material at 20 B, a mid rate and 400 B: trace parity and exact PCM frame by
    frame and time-parallel; decoded output is clipped at both rails somewhere."""
    F = 6
    pcm = E.make_edge_pcm(2 * N_CLS, F, fs, ms)
    clipped = set()
    for nb in (20, 20 + 8 * (_fs_ind(fs, ms) + 2), 400):
        frames = O.encode_streams(pcm, fs, ms, nb)
        lens = np.full(frames.shape[:2], nb, np.int32)
        assert_parity(fs, ms, frames, lens)
        m_pcm, _ = _decode_multi(fs, ms, frames, lens)
        assert_pcm_matches_oracle(m_pcm, fs, ms, frames, lens, (fs, ms, nb, "decode_stream_frames"))
        clipped |= set(np.intersect1d(m_pcm, [32767, -32768]).tolist())
    assert clipped == {32767, -32768}
