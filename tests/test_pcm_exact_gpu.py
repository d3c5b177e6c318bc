"""Decoder PCM to the bit, where synthesis is checked least: concealment fades, post-filter transitions, quiet material,
and every synthesis kernel and entry point.

The gate (tests/common.py assert_pcm_matches_oracle, and assert_parity) is bit equality with the oracle run with the
engine's inverse MDCT (oracle/lc3o_engine_imdct.cpp), whose concealment, overlap-add, post filter and rounding are the
oracle's own code; PCM also stays within +-1 LSB of the oracle run with the reference's transform.  A twiddle, window or
post-filter coefficient wrong in its last bit, or a fade factor off by one ulp, changes some output sample here even
where it stays far below 1 LSB.
"""
import functools

import numpy as np
import pytest

from common import ALL_CONFIGS, assert_parity, assert_pcm_matches_oracle, corpus, corpus_clip, gpu_decode
from oracle import pyoracle as O
from tools import edge_corpus as E
from tools.corpus import MIXED_NBYTES

pytestmark = pytest.mark.gpu

TR_OK, TR_LTPF_ACTIVE, TR_PITCH_INDEX = O.TR["OK"], O.TR["LTPF_ACTIVE"], O.TR["PITCH_INDEX"]


def _decoder(fs, ms, S, nb, synth_mode=0):
    import torch

    import lc3_codec_b200 as L
    sf, fd = L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)
    ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(S, fd, sf, nb), dtype=torch.uint8, device="cuda:0")
    dec = L.Lc3BatchDecoder(S, fd, sf, ws, nb)
    dec.set_synth_mode(synth_mode)
    return dec


def _decode_multi(fs, ms, frames, lens):
    """frames [S, F, nb] -> pcm [S, F, nf] through one lc3b_decode_stream_frames call of a fresh handle."""
    import torch
    S, F, nb = frames.shape
    dec = _decoder(fs, ms, S, nb)
    scratch = torch.empty(dec.multi_scratch_bytes(F), dtype=torch.uint8, device="cuda:0")
    out = torch.zeros((S, F * dec.nf), dtype=torch.int16, device="cuda:0")
    ln = torch.from_numpy(np.ascontiguousarray(lens.astype(np.int32))).cuda()
    dec.decode_stream_frames(16, torch.from_numpy(np.ascontiguousarray(frames)).cuda(), out, scratch, ln)
    torch.cuda.synchronize()
    return out.cpu().numpy().reshape(S, F, dec.nf)


# ------------------------------------------------------------------------------------------------------------ concealment
@pytest.mark.parametrize("fs,ms,nb", [(48000, 10, 100), (16000, 7.5, 30)])
def test_loss_runs_of_every_length(fs, ms, nb):
    """Loss runs of 1 to 20 frames, so the fade goes 1.0 -> 0.9 (from the 5th lost frame) -> 0.85 (from the 9th): on
    streams 0-19 the run ends in a frame whose post filter is active (where the material has one), on streams 20-39 the
    run starts at frame 0, before any good frame.  Frame by frame and time-parallel."""
    S, F, R = 40, 44, 20
    _, frames = corpus(fs, ms, nb, S, F)
    clean_tr = O.decode_streams(frames, fs, ms, trace=True)[1]
    lens = np.full((S, F), nb, np.int32)
    into_active = 0
    for run in range(1, R + 1):
        s = run - 1
        active = np.flatnonzero(clean_tr[s, 4 + run:F - 2, TR_LTPF_ACTIVE]) + 4 + run      # recovery frames on the filter
        end = int(active[0]) if active.size else 4 + run
        into_active += bool(active.size)
        lens[s, end - run:end] = 0
        lens[R + s, :run] = 0
    assert into_active >= R // 2, into_active
    stats = assert_parity(fs, ms, frames, lens)
    assert stats["concealed"] > 0.1
    assert_pcm_matches_oracle(_decode_multi(fs, ms, frames, lens), fs, ms, frames, lens, (fs, ms, "decode_stream_frames"))


# ------------------------------------------------------------------------------------------------------------ post filter
def _transition_cases(tr):
    """Counts of the post filter's five transition cases (long_term_post_filter.rs:252-343) from a trace [S, F, 48];
    concealed frames run with the filter off.  Case 4 is taken as an unchanged pitch index."""
    act = (tr[..., TR_OK] == 1) & (tr[..., TR_LTPF_ACTIVE] == 1)
    cur, prev = act[:, 1:], act[:, :-1]
    same = tr[:, 1:, TR_PITCH_INDEX] == tr[:, :-1, TR_PITCH_INDEX]
    return [int((~cur & ~prev).sum()), int((cur & ~prev).sum()), int((~cur & prev).sum()), int((cur & prev & same).sum()),
            int((cur & prev & ~same).sum())]


@pytest.mark.parametrize("fs,ms,nb", [(48000, 10, 40), (48000, 10, 60), (48000, 10, 80), (48000, 10, 100), (16000, 7.5, 30)])
def test_post_filter_transitions_over_whole_clips(fs, ms, nb):
    """200-frame clips at the rates where the post filter acts, so its state accumulates over the whole clip: all five
    transition cases occur, PCM exact frame by frame and time-parallel."""
    _, frames = corpus_clip(fs, ms, nb, 48)
    lens = np.full(frames.shape[:2], nb, np.int32)
    tr = O.decode_streams(frames, fs, ms, trace=True)[1]
    cases = _transition_cases(tr)
    assert min(cases) > 0, cases
    assert_parity(fs, ms, frames)
    assert_pcm_matches_oracle(_decode_multi(fs, ms, frames, lens), fs, ms, frames, lens, (fs, ms, nb, "decode_stream_frames"))


# ------------------------------------------------------------------------------------------------------------ quiet material
@functools.lru_cache(maxsize=1)
def _quiet_pcm(fs, ms, F):
    silence = E.make_edge_streams(E.streams_of("silence", 2), F, fs, ms)
    dither = E.make_edge_streams(E.streams_of("dither", 4), F, fs, ms)
    return np.concatenate([silence, dither, E.make_quiet_tone_pcm(4, F, fs, ms)])


@pytest.mark.parametrize("fs,ms", ALL_CONFIGS)
def test_quiet_material(fs, ms):
    """Silence, +-1 LSB dither and -90 dBFS tones at the lowest, a middle and the highest rate: decoded samples of
    magnitude 0, 1 and 2, where a +-1 LSB gate checks next to nothing."""
    F = 8
    pcm = _quiet_pcm(fs, ms, F)
    nonzero = 0
    for nb in (20, MIXED_NBYTES[(fs, ms)], 400):
        frames = O.encode_streams(pcm, fs, ms, nb)
        lens = np.full(frames.shape[:2], nb, np.int32)
        assert_parity(fs, ms, frames, lens)
        e_pcm = assert_pcm_matches_oracle(_decode_multi(fs, ms, frames, lens), fs, ms, frames, lens, (fs, ms, nb, "multi"))
        assert (e_pcm[:2] == 0).all()                                   # silence decodes to silence
        nonzero += int(np.count_nonzero(e_pcm[2:]))
    assert nonzero > 0


# ------------------------------------------------------------------------------------------------------------ every kernel
def _pair_min_rows():
    """The smallest launch that runs synth_pair_kernel (as tests/test_synth_regfft_gpu.py)."""
    import torch
    return 2 * torch.cuda.get_device_properties(0).multi_processor_count * 5 * 4 * 2


def _lossy(frames, seed, p_lost=0.1, p_garbage=0.05):
    rng = np.random.default_rng(seed)
    frames = frames.copy()
    S, F, nb = frames.shape
    lens = np.full((S, F), nb, np.int32)
    lens[rng.random((S, F)) < p_lost] = 0
    bad = rng.random((S, F)) < p_garbage
    frames[bad] = rng.integers(0, 256, (int(bad.sum()), nb), dtype=np.uint8)
    return frames, lens


@pytest.mark.parametrize("fs,nb", [(48000, 150), (44100, 130)])
def test_pair_kernel_and_single_frame_kernel(fs, nb):
    """Above the pair threshold (an odd row count): synth mode 0 runs synth_pair_kernel, mode 1 synth_classic_kernel;
    both exact against the oracle, lost and garbage frames included."""
    S = _pair_min_rows() + 1
    _, base = corpus(fs, 10, nb, 64, 3)
    frames, lens = _lossy(np.tile(base, ((S + 63) // 64, 1, 1))[:S], seed=S)
    for mode in (0, 1):
        pcm = gpu_decode(fs, 10, frames, lens, trace=False, synth_mode=mode)[0]
        assert_pcm_matches_oracle(pcm, fs, 10, frames, lens, (fs, "synth mode", mode))


@pytest.mark.parametrize("dequant_mode,graph,split", [(1, True, None), (1, False, None), (2, True, 4), (2, False, 2)])
def test_dequantisation_modes_graph_and_split(dequant_mode, graph, split):
    """Both dequantisation kernels, the graph executor on and off, sub-batches: exact PCM at 48 kHz / 10 ms and 16 kHz /
    7.5 ms with lost and garbage frames."""
    for fs, ms, nb in ((48000, 10, 80), (16000, 7.5, 30)):
        _, clean = corpus(fs, ms, nb, 300, 8)
        frames, lens = _lossy(clean, seed=dequant_mode * 10 + (split or 1))
        assert_parity(fs, ms, frames, lens, dequant_mode=dequant_mode, graph=graph, split=split)


def test_subset_calls_with_ids_in_random_order():
    """lc3b_decode_frames_subset with a random subset of streams in random order per call: each stream decodes its own
    frames in order whenever it is listed; its outputs are exactly the oracle's first frames of that stream."""
    import torch
    fs, ms, nb, S, P = 48000, 10, 60, 200, 12
    _, clean = corpus(fs, ms, nb, S, P)
    frames, lens = _lossy(clean, seed=41)
    dec = _decoder(fs, ms, S, nb)
    rng = np.random.default_rng(43)
    done = np.zeros(S, np.int64)
    got = np.zeros((S, P, dec.nf), np.int16)
    for _ in range(P):
        ids = rng.permutation(S)[:int(rng.integers(S // 3, S + 1))].astype(np.int32)
        ids = ids[done[ids] < P]
        k = done[ids]
        out = torch.zeros((len(ids), dec.nf), dtype=torch.int16, device="cuda:0")
        dec.decode_frames_subset(16, ids, torch.from_numpy(np.ascontiguousarray(frames[ids, k])).cuda(), out,
                                 torch.from_numpy(np.ascontiguousarray(lens[ids, k])).cuda())
        got[ids, k] = out.cpu().numpy()
        done[ids] += 1
    e_pcm = O.decode_streams(frames, fs, ms, lens, transform="engine")
    for s in range(S):
        assert np.array_equal(got[s, :done[s]], e_pcm[s, :done[s]]), s
    assert done.min() > 0 and done.min() < done.max()                 # every stream decoded, some skipped calls


def test_mixed_rate_decoder_at_every_configuration():
    """One Lc3MixedBatchDecoder over all twelve configurations, lost and garbage frames included: every bucket exact."""
    import torch

    import lc3_codec_b200 as L
    per, F = 16, 8
    data = {}
    for k in ALL_CONFIGS:
        _, clean = corpus(*k, MIXED_NBYTES[k], per, F)
        data[k] = _lossy(clean, seed=k[0] + int(2 * k[1]))
    stream_cfg = [ALL_CONFIGS[s % 12] for s in range(12 * per)]
    dec = L.Lc3MixedBatchDecoder([(L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)) for fs, ms in stream_cfg],
                                 max_nbytes=120, device="cuda:0")
    S = len(stream_cfg)
    got = np.zeros((S, F, 480), np.int16)
    for f in range(F):
        rows, lens = np.zeros((S, 120), np.uint8), np.zeros(S, np.int32)
        for pos, s in enumerate(dec.order):
            fr, ln = data[stream_cfg[s]]
            rows[pos, :fr.shape[2]] = fr[s // 12, f]
            lens[pos] = ln[s // 12, f]
        out = torch.zeros((S, 480), dtype=torch.int16, device="cuda:0")
        dec.decode_frames(16, torch.from_numpy(rows).cuda(), torch.from_numpy(lens).cuda(), out)
        torch.cuda.synchronize()
        got[np.array(dec.order), f] = out.cpu().numpy()
    for i, k in enumerate(ALL_CONFIGS):
        fr, ln = data[k]
        assert_pcm_matches_oracle(got[i::12], *k, fr, ln, k)


def test_host_entry_point():
    """lc3b_decode_frames_host, lost and garbage frames included."""
    _, clean = corpus(32000, 7.5, 60, 96, 10)
    frames, lens = _lossy(clean, seed=47)
    assert_parity(32000, 7.5, frames, lens, host=True)
