"""Shared helpers for the parity tests: corpus construction (oracle encoder) and a frame-by-frame GPU driver."""
from __future__ import annotations

import functools

import numpy as np

from oracle import pyoracle as O
from tools.corpus import CLIP_FRAMES, MIXED_NBYTES, clip_offsets, make_pcm, take_window

ALL_CONFIGS = sorted(MIXED_NBYTES.keys())


@functools.lru_cache(maxsize=32)
def corpus(fs: int, ms: float, nbytes: int, n_streams: int, n_frames: int, first_stream: int = 0):
    """(pcm [S,F,nf] i16, frames [S,F,nbytes] u8) - synthetic audio encoded by the ORACLE encoder."""
    cfg = O.config(fs, ms)
    pcm = make_pcm(n_streams, n_frames, fs, cfg["nf"], first_stream)
    frames = O.encode_streams(pcm, fs, ms, nbytes)
    return pcm, frames


@functools.lru_cache(maxsize=2)
def _clip_pcm(fs: int, nf: int, n_streams: int, first_stream: int):
    return make_pcm(n_streams, CLIP_FRAMES, fs, nf, first_stream)


@functools.lru_cache(maxsize=8)
def corpus_clip(fs: int, ms: float, nbytes: int, n_streams: int, window: int = 0, first_stream: int = 0):
    """SURVEY.md 8d clips: 200 frames per stream, oracle-encoded from frame 0.  window = 0 returns the whole clips
    (pcm [S,200,nf], frames [S,200,nbytes]); window = n returns n consecutive frames per stream at the per-stream
    offset of tools.corpus.clip_offsets (in [10, 200 - n]), i.e. what bench.py's fixtures hold."""
    cfg = O.config(fs, ms)
    pcm = _clip_pcm(fs, cfg["nf"], n_streams, first_stream)
    frames = O.encode_streams(pcm, fs, ms, nbytes)
    if window:
        off = clip_offsets(n_streams, window, first_stream)
        return take_window(pcm, off, window), take_window(frames, off, window)
    return pcm, frames


def gpu_decode(fs, ms, frames, nbytes_per_frame=None, host=False, trace=True, device="cuda:0", dequant_mode=0, graph=None,
               min_nbytes=0, synth_mode=0, split=None):
    """Decode [S,F,nbytes] frame by frame through the C ABI; returns pcm [S,F,nf], trace [S,F,48], x [S,F,ne],
    spectrum [S,F,ne], status [S,F]."""
    import torch

    import lc3_codec_b200 as L

    S, F, nb = frames.shape
    sf, fd = L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)
    nbytes_ws = max(nb, 1)
    ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(S, fd, sf, nbytes_ws), dtype=torch.uint8, device=device)
    dec = L.Lc3BatchDecoder(S, fd, sf, ws, nbytes_ws)
    dec.set_dequant_mode(dequant_mode)                  # 0 auto, 1 warp-per-frame kernel, 2 thread-per-frame kernel
    if graph is not None:
        dec.set_graph_mode(graph)
    dec.set_synth_mode(synth_mode)                      # 0 kernel by launch size, 1 one frame per warp always
    if split is not None:
        dec.set_split(split)                            # sub-batches per call (include/lc3b.h)
    if min_nbytes:
        dec.set_min_nbytes(min_nbytes)                  # the handle may drop the post filter's history (include/lc3b.h)
    nf, ne = dec.nf, dec.ne
    pcm = np.zeros((S, F, nf), np.int16)
    tr = np.zeros((S, F, 48), np.int32)
    xs = np.zeros((S, F, ne), np.int32)
    sp = np.zeros((S, F, ne), np.float32)
    status = np.zeros((S, F), np.int32)
    if trace:
        d_tr, d_x = dec.enable_trace()
    for f in range(F):
        fr = torch.from_numpy(np.ascontiguousarray(frames[:, f]))
        ln = None if nbytes_per_frame is None else torch.from_numpy(np.ascontiguousarray(nbytes_per_frame[:, f].astype(np.int32)))
        if host:
            out = torch.zeros((S, nf), dtype=torch.int16).pin_memory()
            st = torch.zeros(S, dtype=torch.int32).pin_memory()
            dec.decode_frames_host(16, fr.pin_memory(), out, None if ln is None else ln.pin_memory(), status_out=st)
            torch.cuda.synchronize()
        else:
            out = torch.zeros((S, nf), dtype=torch.int16, device=device)
            st = torch.zeros(S, dtype=torch.int32, device=device)
            dec.decode_frames(16, fr.to(device), out, None if ln is None else ln.to(device), status_out=st)
        pcm[:, f] = out.cpu().numpy()
        status[:, f] = st.cpu().numpy()
        if trace:
            tr[:, f] = d_tr.cpu().numpy()
            xs[:, f] = d_x.cpu().numpy()
            sp[:, f] = dec.spectrum().cpu().numpy()
    return pcm, tr, xs, sp, status


def assert_pcm_matches_oracle(g_pcm, fs, ms, frames, nbytes_per_frame=None, what=""):
    """The decoder's PCM gates against the oracle on the same bytes: bit exact against the oracle run with the engine's
    inverse MDCT (oracle/lc3o_engine_imdct.cpp; everything else is the oracle's own code), and within +-1 LSB against the
    oracle run with the reference's (the two DCT-IVs differ in their last bits, tests/test_engine_transform_cpu.py).
    g_pcm may be wider than nf.  Returns the reference-transform oracle's PCM."""
    e_pcm = O.decode_streams(frames, fs, ms, nbytes_per_frame, transform="engine")
    o_pcm = O.decode_streams(frames, fs, ms, nbytes_per_frame)
    g = np.asarray(g_pcm)[..., :o_pcm.shape[-1]]
    bad = np.argwhere(g != e_pcm)
    assert bad.size == 0, f"{what}: PCM not bit exact against the engine-transform oracle in {len(bad)} samples, first " \
                          f"(stream, frame, n) {bad[:4].tolist()}: gpu {g[tuple(bad[0])]} oracle {e_pcm[tuple(bad[0])]}"
    d = np.abs(o_pcm.astype(np.int32) - g.astype(np.int32))
    assert d.max() <= 1, f"{what}: PCM differs from the reference transform by {d.max()} LSB at {np.argwhere(d > 1)[:4].tolist()}"
    return o_pcm


def assert_parity(fs, ms, frames, nbytes_per_frame=None, host=False, exact_spectrum=True, dequant_mode=0, graph=None,
                  min_nbytes=0, split=None):
    """The decoder parity gates of SURVEY.md 8d against the oracle on the same bytes, PCM to the bit."""
    o_pcm, o_tr, o_x, o_sp = O.decode_streams(frames, fs, ms, nbytes_per_frame, trace=True)
    e_pcm = O.decode_streams(frames, fs, ms, nbytes_per_frame, transform="engine")
    g_pcm, g_tr, g_x, g_sp, g_status = gpu_decode(fs, ms, frames, nbytes_per_frame, host=host, dequant_mode=dequant_mode, graph=graph,
                                                    min_nbytes=min_nbytes, split=split)
    # (i) side info, TNS data, integer spectrum, residual-bit count, seed, zero-frame flag: bit exact
    bad = np.argwhere(o_tr != g_tr)
    assert bad.size == 0, f"trace mismatch at (stream, frame, word) {bad[:8].tolist()}: " \
                          f"oracle {o_tr[tuple(bad[0])]} gpu {g_tr[tuple(bad[0])]}"
    assert np.array_equal(o_x, g_x), f"integer spectrum differs in {np.count_nonzero((o_x != g_x).any(-1))} frames"
    assert np.array_equal(g_status, 1 - o_tr[..., 0])
    # the shaped spectrum handed to the IMDCT is computed with contraction-free f32 ops in the reference's
    # order: bit exact on decoded frames (concealed frames hold the last good spectrum in the GPU slot)
    if exact_spectrum:
        ok = o_tr[..., 0] == 1
        assert np.array_equal(o_sp[ok].view(np.uint32), g_sp[ok].view(np.uint32)), "shaped spectrum not bit exact"
    # (ii) PCM bit exact against the oracle with the engine's inverse MDCT: concealment, overlap-add, post filter and
    # rounding are the oracle's, so only the transform separates the two gates below
    bad = np.argwhere(g_pcm != e_pcm)
    assert bad.size == 0, f"PCM not bit exact against the engine-transform oracle in {len(bad)} samples, first (stream, " \
                          f"frame, n) {bad[:4].tolist()}: gpu {g_pcm[tuple(bad[0])]} oracle {e_pcm[tuple(bad[0])]}"
    # (iii) PCM within +-1 LSB against the reference's transform (kissfft DCT-IV)
    d = np.abs(o_pcm.astype(np.int32) - g_pcm.astype(np.int32))
    assert d.max() <= 1, f"PCM differs by {d.max()} LSB (streams {np.unique(np.argwhere(d > 1)[:, 0])[:8]})"
    return dict(pcm_exact=float((d == 0).mean()), concealed=float((o_tr[..., 0] == 0).mean()),
                lsb_mode=float(o_tr[..., 3].mean()), ltpf_active=float(o_tr[..., 18].mean()),
                tns=float((o_tr[..., 21] > 0).mean()),
                mean_lastnz=float(o_tr[..., 2][o_tr[..., 0] == 1].mean()) if (o_tr[..., 0] == 1).any() else 0.0,
                near_empty=float((o_tr[..., 2][o_tr[..., 0] == 1] <= 16).mean()) if (o_tr[..., 0] == 1).any() else 0.0)


def gpu_encode(fs, ms, pcm, nbytes, host=False, device="cuda:0", debug=False):
    """Encode [S,F,nf] i16 frame by frame through the C ABI -> bytes [S,F,nbytes] (+ per-frame intermediates if debug)."""
    import torch

    import lc3_codec_b200 as L

    S, F, nf = pcm.shape
    sf, fd = L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)
    ws = torch.empty(L.Lc3BatchEncoder.calc_working_buffer_lengths(S, fd, sf, nbytes), dtype=torch.uint8, device=device)
    enc = L.Lc3BatchEncoder(S, fd, sf, ws, nbytes)
    out = np.zeros((S, F, nbytes), np.uint8)
    dbg = []
    for f in range(F):
        x = torch.from_numpy(np.ascontiguousarray(pcm[:, f]))
        if host:
            y = torch.zeros((S, nbytes), dtype=torch.uint8).pin_memory()
            enc.encode_frames_host(x.pin_memory(), y)
            torch.cuda.synchronize()
        else:
            y = torch.zeros((S, nbytes), dtype=torch.uint8, device=device)
            enc.encode_frames(x.to(device), y)
        out[:, f] = y.cpu().numpy()
        if debug:
            dbg.append([t.cpu().numpy() for t in enc.debug_read()])
    return (out, dbg) if debug else out


def snr_db(ref, test):
    ref = ref.astype(np.float64)
    err = ref - test.astype(np.float64)
    return 10.0 * np.log10((ref ** 2).sum() / max((err ** 2).sum(), 1e-30))


def codec_delay(pcm, dec_pcm):
    """Delay D (samples) at which the decoder's output lines up with the encoder's input: dec[t] ~ in[t - D].
    Found by minimising the mean squared error over D in [0, nf) on the streams given (LC3: nf - 2 z, the 2.5 ms
    look-ahead at 10 ms frames; the frame period itself is hidden by feeding frame f in and reading frame f out)."""
    S, F, nf = pcm.shape
    x = pcm.reshape(S, -1).astype(np.float64)
    y = dec_pcm.reshape(S, -1).astype(np.float64)
    errs = [((y[:, d:] - x[:, :x.shape[1] - d]) ** 2).mean() for d in range(0, nf)]
    return int(np.argmin(errs))


def encoder_gate(pcm, o_frames, g_frames, fs, ms, min_identical=0.999, snr_tol_db=0.1):
    """Encoder parity gate (SURVEY.md 8d iii, BASELINE.json north_star): bitstreams byte-identical on at least
    `min_identical` of the frames, and EVERY differing frame decodes (oracle decoder, each bitstream set decoded as a
    whole so the overlap of the neighbouring frames is the set's own) to an SNR against the delayed input that is
    within `snr_tol_db` of the oracle frame's.  Pure CPU; returns (identical fraction, worst |dSNR| in dB)."""
    same = (o_frames == g_frames).all(-1)
    frac = float(same.mean())
    worst = 0.0
    if not same.all():
        S, F, nf = pcm.shape
        o_pcm = O.decode_streams(o_frames, fs, ms)
        g_pcm = O.decode_streams(g_frames, fs, ms)
        D = codec_delay(pcm, o_pcm)
        x = np.concatenate([np.zeros((S, D), np.int16), pcm.reshape(S, -1)], axis=1)[:, :F * nf].reshape(S, F, nf)
        for s, f in np.argwhere(~same):
            ref = x[s, f].astype(np.float64)
            if (ref ** 2).sum() < 1.0:                  # silent input: SNR undefined, the two decodes must both be silent-ish
                assert np.abs(o_pcm[s, f].astype(np.int32) - g_pcm[s, f].astype(np.int32)).max() <= 2, (s, f)
                continue
            d_snr = abs(snr_db(ref, g_pcm[s, f]) - snr_db(ref, o_pcm[s, f]))
            worst = max(worst, d_snr)
            assert d_snr <= snr_tol_db, f"stream {s} frame {f}: bytes differ and decoded SNR differs by {d_snr:.3f} dB"
    assert frac >= min_identical, f"only {frac * 100:.3f} % of frames byte-identical " \
                                  f"(first mismatches at {np.argwhere(~same)[:5].tolist()})"
    return frac, worst


def assert_encoder_parity(fs, ms, nbytes, n_streams, n_frames, host=False, min_identical=0.999, clip=False):
    """GPU encoder vs oracle encoder on the same PCM through encoder_gate().  clip=True: 200-frame SURVEY 8d clips
    (n_frames ignored)."""
    pcm, o_frames = corpus_clip(fs, ms, nbytes, n_streams) if clip else corpus(fs, ms, nbytes, n_streams, n_frames)
    g_frames = gpu_encode(fs, ms, pcm, nbytes, host=host)
    return encoder_gate(pcm, o_frames, g_frames, fs, ms, min_identical)[0]
