"""GPU parity tests for the decode path: CUDA engine (through the C ABI) vs the CPU oracle on the same bytes.

Parity bar (BASELINE.json north_star / SURVEY.md 8d):
  * entropy-decoded integer spectrum and side info: bit exact;
  * decoded i16 PCM: within +-1 LSB (PCM_TOL below);
  * reference golden vector lc3_decode_channel: +-1 LSB (the engine's FFT factorisation differs from kissfft).
Run on the B200 box: python -m pytest tests -m gpu
"""
import numpy as np
import pytest

from common import ALL_CONFIGS, assert_parity, corpus, corpus_clip, gpu_decode
from conftest import load_golden
from tools.corpus import MIXED_NBYTES

pytestmark = pytest.mark.gpu
PCM_TOL = 1


def test_golden_lc3_decode_channel():
    """src/decoder/lc3_decoder.rs:374 - the reference's own end-to-end vector, replicated over 33 streams."""
    buf, exp = load_golden("decoder__lc3_decoder__lc3_decode_channel")
    frames = np.tile(np.array(buf, np.uint8)[None, None, :], (33, 1, 1))
    pcm, tr, x, sp, st = gpu_decode(48000, 10, frames)
    assert (st == 0).all()
    d = np.abs(pcm[:, 0].astype(np.int32) - exp[None, :].astype(np.int32))
    assert d.max() <= PCM_TOL
    assert (pcm == pcm[:1]).all()                       # every lane decodes identically
    # arithmetic_codec.rs:458-473 scalars of the same frame
    assert tr[0, 0, 40] == 56909 and tr[0, 0, 21] == 8 and tr[0, 0, 22] == 0
    assert tr[0, 0, 23:39].tolist() == [6, 10, 7, 8, 7, 9, 7, 7, 0, 0, 0, 0, 0, 0, 0, 0]
    _, xi, _ = load_golden("decoder__noise_filling__decode_noise_filling")
    assert np.array_equal(x[0, 0], xi)


def test_c1_48k_10ms_150B():
    """BASELINE config 1/5 shape: 48 kHz, 10 ms, 150 B (lsb_mode frames occur, LTPF gain 0)."""
    _, frames = corpus(48000, 10, 150, 160, 24)
    stats = assert_parity(48000, 10, frames)
    assert stats["concealed"] == 0.0
    assert stats["lsb_mode"] > 0.0 and stats["tns"] > 0.0, stats


def test_c3_16k_7p5ms_30B_ltpf_active():
    """BASELINE config 3: 16 kHz, 7.5 ms, 30 B - LTPF and TNS active, 3-block histories."""
    _, frames = corpus(16000, 7.5, 30, 192, 48)
    stats = assert_parity(16000, 7.5, frames)
    assert stats["ltpf_active"] > 0.0, stats


@pytest.mark.parametrize("fs,ms", ALL_CONFIGS)
def test_all_rates_and_durations(fs, ms):
    """BASELINE config 4's twelve (fs, duration) combinations at their mixed-rate byte sizes."""
    if fs == 8000:
        pytest.skip("reference encoder cannot be constructed at 8 kHz (bandwidth_detector.rs:42); covered below")
    _, frames = corpus(fs, ms, MIXED_NBYTES[(fs, ms)], 96, 30)
    assert_parity(fs, ms, frames)


@pytest.mark.parametrize("ms", [7.5, 10])
def test_8k_streams(ms):
    """8 kHz bitstreams come from the oracle encoder with the spec's 8 kHz handling (see DESIGN.md)."""
    _, frames = corpus(8000, ms, MIXED_NBYTES[(8000, ms)], 64, 30)
    assert_parity(8000, ms, frames)


@pytest.mark.parametrize("nbytes", [40, 60, 80, 100])
def test_48k_low_rates_ltpf(nbytes):
    """48 kHz 10 ms below 880 bits: LTPF gains 0.4 .. 0.25 and all five transition cases occur on speech-like streams."""
    _, frames = corpus(48000, 10, nbytes, 96, 60)
    assert_parity(48000, 10, frames)


def test_lost_and_corrupt_frames():
    """Concealment parity (packet_loss_concealment.rs:63): dropped frames (len 0), runs longer than 8, bit flips."""
    _, frames = corpus(48000, 10, 100, 96, 40)
    frames = frames.copy()
    S, F, nb = frames.shape
    rng = np.random.default_rng(7)
    lens = np.full((S, F), nb, np.int32)
    lens[rng.random((S, F)) < 0.08] = 0
    lens[5, 10:24] = 0                                   # long loss: alpha fades 0.9 then 0.85
    lens[6, 0:3] = 0                                     # loss before any good frame
    flip = rng.random((S, F)) < 0.10
    for s, f in np.argwhere(flip):
        for _ in range(int(rng.integers(1, 6))):
            frames[s, f, rng.integers(0, nb)] ^= 1 << int(rng.integers(0, 8))
    stats = assert_parity(48000, 10, frames, lens)
    assert stats["concealed"] > 0.05


def test_garbage_frames():
    """Uniformly random bytes: exercises every error exit of side_info_reader / arithmetic_codec and the lev == 14 quirk."""
    rng = np.random.default_rng(11)
    for fs, ms, nb in ((48000, 10, 150), (16000, 7.5, 30), (32000, 10, 80)):
        frames = rng.integers(0, 256, size=(128, 12, nb), dtype=np.uint8)
        assert_parity(fs, ms, frames)


def test_variable_frame_lengths():
    """buf_in.len() may change per call and per stream (lc3_decoder.rs:85): shorter frames inside a wider stride."""
    _, f150 = corpus(48000, 10, 150, 64, 16)
    _, f60 = corpus(48000, 10, 60, 64, 16)
    frames = f150.copy()
    lens = np.full((64, 16), 150, np.int32)
    sel = (np.arange(64)[:, None] + np.arange(16)[None, :]) % 3 == 0
    frames[sel, :60] = f60[sel]
    frames[sel, 60:] = 0xAA
    lens[sel] = 60
    # the oracle is handed each frame at its own length: compare against per-length decodes
    from oracle import pyoracle as O
    o_pcm, o_tr, o_x, _ = O.decode_streams(frames, 48000, 10, lens, trace=True)
    g_pcm, g_tr, g_x, _, _ = gpu_decode(48000, 10, frames, lens)
    assert np.array_equal(o_tr, g_tr) and np.array_equal(o_x, g_x)
    assert np.abs(o_pcm.astype(np.int32) - g_pcm.astype(np.int32)).max() <= PCM_TOL


def test_host_buffer_entry_point():
    """lc3b_decode_frames_host: pinned host buffers in, host PCM out, same results."""
    _, frames = corpus(24000, 10, 60, 70, 10)
    assert_parity(24000, 10, frames, host=True)


def test_pipelined_host_entry_point():
    """lc3b_decoder_set_host_pipelining: PCM copies overlap the next call's kernels; results are unchanged."""
    import torch

    import lc3_codec_b200 as L
    from oracle import pyoracle as O
    _, frames = corpus(48000, 10, 100, 70, 12)
    S, F, nb = frames.shape
    sf, fd = L.SamplingFrequency.Hz48000, L.FrameDuration.TenMs
    ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(S, fd, sf, nb), dtype=torch.uint8, device="cuda:0")
    dec = L.Lc3BatchDecoder(S, fd, sf, ws, nb)
    dec.set_host_pipelining(True)
    host_in = torch.from_numpy(np.ascontiguousarray(frames.transpose(1, 0, 2))).pin_memory()      # [F,S,nb]
    host_out = torch.zeros((F, S, 480), dtype=torch.int16).pin_memory()
    for f in range(F):
        dec.decode_frames_host(16, host_in[f], host_out[f])
    dec.host_fence()
    torch.cuda.synchronize()
    o_pcm = O.decode_streams(frames, 48000, 10)
    d = np.abs(host_out.numpy().transpose(1, 0, 2).astype(np.int32) - o_pcm.astype(np.int32))
    assert d.max() <= PCM_TOL


def test_odd_pcm_stride_and_unaligned_rows():
    """pcm_out rows at an odd sample pitch / 2-byte-aligned base take the kernels' scalar store path; same samples."""
    import torch

    import lc3_codec_b200 as L
    for fs, ms, nb in ((48000, 10, 150), (16000, 7.5, 30)):
        _, frames = corpus(fs, ms, nb, 40, 6)
        ref = gpu_decode(fs, ms, frames, trace=False)[0]
        sf, fd = L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)
        ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(40, fd, sf, nb), dtype=torch.uint8, device="cuda:0")
        dec = L.Lc3BatchDecoder(40, fd, sf, ws, nb)
        nf = dec.nf
        backing = torch.zeros(40 * (nf + 3) + 1, dtype=torch.int16, device="cuda:0")
        out = backing[1:].view(40, nf + 3)[:, :nf + 1]         # base 2-byte aligned only, pitch nf + 3 (odd)
        for f in range(6):
            dec.decode_frames(16, torch.from_numpy(np.ascontiguousarray(frames[:, f])).cuda(), out)
            assert np.array_equal(out[:, :nf].cpu().numpy(), ref[:, f])
        assert int(out[:, nf].abs().max()) == 0                 # nothing written past nf


def test_ragged_stream_counts():
    """Stream counts that are not multiples of the warp / CTA sizes."""
    for n in (1, 31, 33, 129):
        _, frames = corpus(32000, 7.5, 60, n, 6)
        assert_parity(32000, 7.5, frames)


def test_only_16_bits_per_sample():
    """lc3_decoder.rs:80: the one error the reference returns."""
    import torch

    import lc3_codec_b200 as L
    ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(4, L.FrameDuration.TenMs, L.SamplingFrequency.Hz48000, 150),
                     dtype=torch.uint8, device="cuda:0")
    dec = L.Lc3BatchDecoder(4, L.FrameDuration.TenMs, L.SamplingFrequency.Hz48000, ws, 150)
    fr = torch.zeros((4, 150), dtype=torch.uint8, device="cuda:0")
    out = torch.zeros((4, 480), dtype=torch.int16, device="cuda:0")
    with pytest.raises(L.Lc3DecoderError):
        dec.decode_frames(24, fr, out)
    with pytest.raises(L.Lc3bError):
        dec.decode_frames(16, fr, out[:, :100])          # short output slice: the reference would truncate/panic


def test_mixed_rate_batch():
    """BASELINE config 4 at test size: all twelve (fs, duration) configurations decoded by one mixed-rate call per frame."""
    import torch

    import lc3_codec_b200 as L
    from oracle import pyoracle as O
    per, F = 24, 10
    cfgs, frames_by, pcm_by = [], {}, {}
    for (fs, ms) in ALL_CONFIGS:
        _, fr = corpus(fs, ms, MIXED_NBYTES[(fs, ms)], per, F)
        frames_by[(fs, ms)] = fr
        pcm_by[(fs, ms)] = O.decode_streams(fr, fs, ms)
    # interleave the configurations over stream ids like SURVEY.md 8d: stream s -> config s mod 12
    stream_cfg = [ALL_CONFIGS[s % 12] for s in range(12 * per)]
    dec = L.Lc3MixedBatchDecoder([(L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)) for fs, ms in stream_cfg],
                                 max_nbytes=120, device="cuda:0")
    S = len(stream_cfg)
    got = np.zeros((S, F, 480), np.int16)
    for f in range(F):
        rows = np.zeros((S, 120), np.uint8)
        lens = np.zeros(S, np.int32)
        for pos, s in enumerate(dec.order):
            fs, ms = stream_cfg[s]
            fr = frames_by[(fs, ms)][s // 12, f]
            rows[pos, :len(fr)] = fr
            lens[pos] = len(fr)
        out = torch.zeros((S, 480), dtype=torch.int16, device="cuda:0")
        dec.decode_frames(16, torch.from_numpy(rows).cuda(), torch.from_numpy(lens).cuda(), out)
        torch.cuda.synchronize()
        got[:, f] = out.cpu().numpy()
    for pos, s in enumerate(dec.order):
        fs, ms = stream_cfg[s]
        exp = pcm_by[(fs, ms)][s // 12]
        nf = exp.shape[-1]
        assert np.abs(got[pos, :, :nf].astype(np.int32) - exp.astype(np.int32)).max() <= PCM_TOL, (fs, ms, s)


def test_mixed_rate_batch_host_entry():
    """lc3b_mixed_decode_frames_host: pinned host rows in, ONE dense pinned PCM buffer out (per-bucket views), pipelined
    copies, status flags; same PCM as the oracle.  Run with the graph executor and with plain launches."""
    import torch

    import lc3_codec_b200 as L
    from oracle import pyoracle as O
    per, F = 10, 6
    frames_by, pcm_by = {}, {}
    for (fs, ms) in ALL_CONFIGS:
        _, fr = corpus(fs, ms, MIXED_NBYTES[(fs, ms)], per, F)
        frames_by[(fs, ms)] = fr
        pcm_by[(fs, ms)] = O.decode_streams(fr, fs, ms)
    stream_cfg = [ALL_CONFIGS[s % 12] for s in range(12 * per)]
    for graph in (True, False):
        dec = L.Lc3MixedBatchDecoder([(L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)) for fs, ms in stream_cfg],
                                     max_nbytes=120, device="cuda:0")
        dec.set_graph_mode(graph)
        dec.set_host_pipelining(True)
        S = len(stream_cfg)
        outs = [dec.alloc_host_pcm() for _ in range(F)]
        status = torch.full((F, S), -1, dtype=torch.int32).pin_memory()
        rows_all = torch.zeros((F, S, 120), dtype=torch.uint8).pin_memory()
        lens = torch.zeros(S, dtype=torch.int32).pin_memory()
        for pos, s in enumerate(dec.order):
            fs, ms = stream_cfg[s]
            fr = frames_by[(fs, ms)][s // 12]
            rows_all[:, pos, :fr.shape[1]] = torch.from_numpy(fr)
            lens[pos] = fr.shape[1]
        for f in range(F):
            dec.decode_frames_host(16, rows_all[f], lens, outs[f], status_out=status[f])
        dec.host_fence()
        torch.cuda.synchronize()
        assert int(status.abs().max()) == 0
        views = [dec.host_pcm_views(o) for o in outs]
        for b, ((sf, fd), first, count) in enumerate(dec.buckets):
            for r in range(count):
                s = dec.order[first + r]
                fs, ms = stream_cfg[s]
                exp = pcm_by[(fs, ms)][s // 12]
                got = np.stack([views[f][b][r].numpy() for f in range(F)])
                assert np.abs(got.astype(np.int32) - exp.astype(np.int32)).max() <= PCM_TOL, (fs, ms, s, graph)


def test_mixed_rate_matches_single_configuration_handles_bitwise():
    """The mixed-rate kernels run the single-configuration bodies: a bucket's PCM must equal, bit for bit, what an
    ordinary lc3b_decode_frames handle produces for the same streams (ragged bucket sizes, lost frames included)."""
    import torch

    import lc3_codec_b200 as L
    sizes = {(48000, 10): 130, (16000, 7.5): 33, (24000, 10): 1, (44100, 7.5): 129, (8000, 10): 40, (32000, 7.5): 64}
    F = 8
    stream_cfg, local = [], []
    for i in range(max(sizes.values())):
        for cfg, n in sizes.items():
            if i < n:
                stream_cfg.append(cfg)
                local.append(i)
    frames_by = {cfg: corpus(cfg[0], cfg[1], MIXED_NBYTES[cfg], n, F)[1] for cfg, n in sizes.items()}
    rng = np.random.default_rng(3)
    lost = {cfg: rng.random((n, F)) < 0.1 for cfg, n in sizes.items()}
    ref = {}
    for cfg, fr in frames_by.items():
        lens = np.where(lost[cfg], 0, fr.shape[2]).astype(np.int32)
        ref[cfg] = gpu_decode(cfg[0], cfg[1], fr, lens, trace=False)
    dec = L.Lc3MixedBatchDecoder([(L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)) for fs, ms in stream_cfg],
                                 max_nbytes=120, device="cuda:0")
    S = len(stream_cfg)
    for f in range(F):
        rows = np.zeros((S, 128), np.uint8)
        lens = np.zeros(S, np.int32)
        for pos, s in enumerate(dec.order):
            cfg = stream_cfg[s]
            fr = frames_by[cfg][local[s], f]
            rows[pos, :len(fr)] = fr
            lens[pos] = 0 if lost[cfg][local[s], f] else len(fr)
        out = torch.zeros((S, 480), dtype=torch.int16, device="cuda:0")
        st = torch.full((S,), -1, dtype=torch.int32, device="cuda:0")
        dec.decode_frames(16, torch.from_numpy(rows).cuda(), torch.from_numpy(lens).cuda(), out, status_out=st)
        got, gst = out.cpu().numpy(), st.cpu().numpy()
        for pos, s in enumerate(dec.order):
            cfg = stream_cfg[s]
            pcm, _, _, _, status = ref[cfg]
            nf = pcm.shape[-1]
            assert np.array_equal(got[pos, :nf], pcm[local[s], f]), (cfg, s, f)
            assert gst[pos] == status[local[s], f]


def test_graph_executor_equals_plain_launches():
    """lc3b_decoder_set_graph_mode: the cached-graph executor replays / patches graphs as the caller's buffers rotate;
    PCM and status are identical to plain launches, and the cache statistics show replays and in-place updates."""
    import torch

    import lc3_codec_b200 as L
    _, frames = corpus(16000, 7.5, 30, 96, 40)
    S, F, nb = frames.shape
    sf, fd = L.SamplingFrequency.Hz16000, L.FrameDuration.SevenPointFiveMs
    outs = []
    for graph in (False, True):
        ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(S, fd, sf, nb), dtype=torch.uint8, device="cuda:0")
        dec = L.Lc3BatchDecoder(S, fd, sf, ws, nb)
        dec.set_graph_mode(graph)
        ring = [torch.zeros((S, nb), dtype=torch.uint8, device="cuda:0") for _ in range(3)]     # caller rotates 3 input buffers
        fresh = []                                                                                # ... then uses new ones every call
        pcm = torch.zeros((F, S, dec.nf), dtype=torch.int16, device="cuda:0")
        for f in range(F):
            if f < 20:
                buf = ring[f % 3]
            else:
                buf = torch.zeros((S, nb), dtype=torch.uint8, device="cuda:0")
                fresh.append(buf)
            buf.copy_(torch.from_numpy(np.ascontiguousarray(frames[:, f])))
            dec.decode_frames(16, buf, pcm[f])
        torch.cuda.synchronize()
        outs.append(pcm.cpu().numpy())
        if graph:
            st = dec.graph_stats()
            assert st["hits"] + st["updates"] + st["builds"] == F and st["builds"] <= 24, st
    assert np.array_equal(outs[0], outs[1])


def test_sharded_decoder_two_shards_on_one_gpu():
    """lc3b_sharded_decoder_*: one host-buffer call for the whole batch, one thread + stream + workspace per shard.
    Two shards on device 0 exercise the row arithmetic and the worker threads on a single-GPU box."""
    import torch

    import lc3_codec_b200 as L
    from oracle import pyoracle as O
    _, frames = corpus(48000, 10, 100, 101, 12)
    S, F, nb = frames.shape
    rng = np.random.default_rng(5)
    lens = np.where(rng.random((S, F)) < 0.1, 0, nb).astype(np.int32)
    dec = L.Lc3ShardedBatchDecoder(S, L.FrameDuration.TenMs, L.SamplingFrequency.Hz48000, nb, devices=[0, 0])
    sh = dec.shards()
    assert [d for d, _, _ in sh] == [0, 0] and sh[0][1] == 0 and sh[0][2] + sh[1][2] == S and sh[1][1] == sh[0][2]
    host_in = torch.from_numpy(np.ascontiguousarray(frames.transpose(1, 0, 2))).pin_memory()
    host_len = torch.from_numpy(np.ascontiguousarray(lens.T)).pin_memory()
    host_out = torch.zeros((F, S, 480), dtype=torch.int16).pin_memory()
    status = torch.full((F, S), -1, dtype=torch.int32).pin_memory()
    for f in range(F):
        dec.decode_frames_host(16, host_in[f], host_out[f], frame_nbytes=host_len[f], status_out=status[f])
    dec.wait()
    o_pcm, o_tr, _, _ = O.decode_streams(frames, 48000, 10, lens, trace=True)
    d = np.abs(host_out.numpy().transpose(1, 0, 2).astype(np.int32) - o_pcm.astype(np.int32))
    assert d.max() <= PCM_TOL
    assert np.array_equal(status.numpy().T, 1 - o_tr[..., 0])
    with pytest.raises(L.Lc3DecoderError):
        dec.decode_frames_host(24, host_in[0], host_out[0])


@pytest.mark.parametrize("mode", [1, 2])
def test_both_dequantisation_kernels_against_the_oracle(mode):
    """lc3b_decoder_set_dequant_mode: the warp-per-frame kernel (small batches) and the thread-per-frame kernel (large
    batches) each meet the full parity bar - shaped spectrum bit exact - on every kind of frame: high-rate frames with
    lsb_mode, TNS with one and two filters, 7.5 ms (window 2), 8 kHz / 7.5 ms (nb = 60 folding), lost frames, garbage."""
    rng = np.random.default_rng(17)
    for fs, ms, nb, S, F in ((48000, 10, 150, 70, 24), (48000, 10, 400, 33, 8), (16000, 7.5, 30, 129, 30), (8000, 7.5, 20, 40, 20),
                             (32000, 7.5, 60, 64, 16), (24000, 10, 60, 31, 16), (44100, 10, 120, 32, 12)):
        _, frames = corpus(fs, ms, nb, S, F)
        lens = np.where(rng.random((S, F)) < 0.06, 0, nb).astype(np.int32)
        stats = assert_parity(fs, ms, frames, lens, dequant_mode=mode, graph=bool(mode & 1))
        assert stats["concealed"] > 0.0
    for fs, ms, nb in ((48000, 10, 150), (16000, 7.5, 30), (8000, 10, 26)):
        frames = rng.integers(0, 256, size=(96, 10, nb), dtype=np.uint8)
        assert_parity(fs, ms, frames, dequant_mode=mode)


def test_dequantisation_kernels_agree_bitwise_at_batch_sizes_around_the_switch():
    """Same streams through mode 1 and mode 2 at 4 096 streams: identical spectra and PCM (tiled corpus)."""
    _, base = corpus(48000, 10, 150, 128, 6)
    frames = np.tile(base, (32, 1, 1))
    a = gpu_decode(48000, 10, frames, dequant_mode=1)
    b = gpu_decode(48000, 10, frames, dequant_mode=2)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[3].view(np.uint32), b[3].view(np.uint32))
    assert np.array_equal(a[1], b[1]) and np.array_equal(a[4], b[4])


def test_min_nbytes_promise_drops_the_post_filter_history_without_changing_results():
    """lc3b_decoder_set_min_nbytes: at >= 110 bytes (48 kHz / 10 ms: 880 bits = 560 + 80 * 4) the reference's gain table row
    is (0.0, 0), so the post filter can never act and its history is dead state.  With the promise the decoder stops
    keeping it; every parity gate still holds - fixed 150 B frames, lengths varying in [110, 150] per call and stream,
    lost frames - and frames that break the promise are concealed / rejected."""
    import torch

    import lc3_codec_b200 as L
    from oracle import pyoracle as O
    _, f150 = corpus(48000, 10, 150, 96, 24)
    assert_parity(48000, 10, f150, min_nbytes=110)
    _, f110 = corpus(48000, 10, 110, 96, 24)
    _, f128 = corpus(48000, 10, 128, 96, 24)
    frames = f150.copy()
    lens = np.full((96, 24), 150, np.int32)
    pick = (np.arange(96)[:, None] * 7 + np.arange(24)[None, :] * 3) % 5
    for val, src, nb in ((1, f110, 110), (2, f128, 128)):
        sel = pick == val
        frames[sel, :nb] = src[sel]
        frames[sel, nb:] = 0x55
        lens[sel] = nb
    lens[pick == 3] = np.broadcast_to(np.where(np.arange(24)[None, :] % 4 == 0, 0, 150), (96, 24))[pick == 3]     # some lost frames
    stats = assert_parity(48000, 10, frames, lens, min_nbytes=110)
    assert stats["concealed"] > 0.0
    # a frame shorter than the promise is treated as lost: same output as handing the decoder an empty slice
    short = lens.copy()
    short[pick == 1] = 60
    as_lost = lens.copy()
    as_lost[pick == 1] = 0
    got = gpu_decode(48000, 10, frames, short, trace=False, min_nbytes=110)
    exp = gpu_decode(48000, 10, frames, as_lost, trace=False, min_nbytes=110)
    assert np.array_equal(got[0], exp[0]) and np.array_equal(got[4], exp[4]) and got[4][pick == 1].all()
    # a promise that does not rule the filter out changes nothing: LTPF stays on at 60 bytes
    _, f60 = corpus(48000, 10, 60, 96, 40)
    stats = assert_parity(48000, 10, f60, min_nbytes=60)
    assert stats["ltpf_active"] > 0.1
    # fixed frame length below the promise: rejected like any other bad argument
    ws = torch.empty(L.Lc3BatchDecoder.calc_working_buffer_lengths(4, L.FrameDuration.TenMs, L.SamplingFrequency.Hz48000, 150),
                     dtype=torch.uint8, device="cuda:0")
    dec = L.Lc3BatchDecoder(4, L.FrameDuration.TenMs, L.SamplingFrequency.Hz48000, ws, 150)
    dec.set_min_nbytes(110)
    with pytest.raises(L.Lc3bError):
        dec.decode_frames(16, torch.zeros((4, 100), dtype=torch.uint8, device="cuda:0"), torch.zeros((4, 480), dtype=torch.int16, device="cuda:0"))
    with pytest.raises(L.Lc3bError):
        dec.set_min_nbytes(151)


@pytest.mark.parametrize("fs,ms,nbytes,split,graph,host", [
    (48000, 10.0, 150, 4, False, False), (48000, 10.0, 150, 2, True, False), (16000, 7.5, 30, 4, False, True),
    (16000, 7.5, 30, 2, True, True)])
def test_sub_batches_match_the_oracle(fs, ms, nbytes, split, graph, host):
    """lc3b_decoder_set_split: a call cut into 2 / 4 sub-batches whose kernels run on the handle's auxiliary streams (or as
    parallel branches of the call's graph).  Ragged on purpose: 700 streams are sub-batches of 256 + 256 + 188 (+ none) or
    384 + 316 - the last one ends in a partly filled CTA.  All three gates against the oracle, lost and short frames
    included, through the device and the host entry points; the thread-per-frame dequantisation kernel is forced because
    the small-batch kernels are never split."""
    _, frames = corpus_clip(fs, ms, nbytes, 700, window=6)
    lens = np.full(frames.shape[:2], nbytes, np.int32)
    rng = np.random.default_rng(5)
    lens[rng.random(lens.shape) < 0.03] = 0                                # lost frames
    stats = assert_parity(fs, ms, frames, lens, host=host, dequant_mode=2, graph=graph, split=split)
    assert stats["concealed"] > 0.0


def test_sub_batches_are_bit_identical_to_one_batch():
    """Same handle configuration, split 1 against split 4, device entry point: PCM, status and the inspection records agree
    bit for bit over consecutive frames (per-stream state carries over between calls in every sub-batch)."""
    _, frames = corpus_clip(48000, 10.0, 150, 1100, window=5)
    a = gpu_decode(48000, 10.0, frames, dequant_mode=2, split=1)
    b = gpu_decode(48000, 10.0, frames, dequant_mode=2, split=4)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
