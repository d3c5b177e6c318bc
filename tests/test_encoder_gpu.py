"""GPU parity tests for the encode path: CUDA engine (through the C ABI) vs the CPU oracle on the same PCM.

Parity bar (BASELINE.json north_star): encoder bitstreams byte-identical on >= 99.9 % of frames.  The engine performs
every decision-feeding f32 operation in the reference's order without FMA, so in practice 100 % is expected.
Run on the B200 box: python -m pytest tests -m gpu
"""
import numpy as np
import pytest

from common import assert_encoder_parity, corpus, gpu_encode
from conftest import load_golden
from tools.corpus import MIXED_NBYTES

pytestmark = pytest.mark.gpu


def test_golden_lc3_encode_channel():
    """src/encoder/lc3_encoder.rs:314 - the reference's own end-to-end vector (first frame of a zero-state encoder)."""
    x, exp = load_golden("encoder__lc3_encoder__lc3_encode_channel")
    pcm = np.tile(x.astype(np.int16)[None, None, :], (5, 1, 1))
    out = gpu_encode(48000, 10, pcm, 150)
    assert np.array_equal(out[0, 0], exp.astype(np.uint8))
    assert (out == out[:1]).all()


def test_c2_48k_10ms_120B():
    """BASELINE config 2 shape: 48 kHz, 10 ms, 120 bytes per channel (attack detector active, LTPF bit off)."""
    assert assert_encoder_parity(48000, 10, 120, 128, 40) == 1.0


def test_c1_48k_10ms_150B():
    assert assert_encoder_parity(48000, 10, 150, 96, 30) == 1.0


def test_16k_7p5ms_30B():
    """BASELINE config 3's encoder side: LTPF decisions, TNS with lpc weighting."""
    assert assert_encoder_parity(16000, 7.5, 30, 128, 60) == 1.0


@pytest.mark.parametrize("fs,ms", [k for k in sorted(MIXED_NBYTES) if k[0] != 8000])
def test_all_rates_and_durations(fs, ms):
    assert assert_encoder_parity(fs, ms, MIXED_NBYTES[(fs, ms)], 64, 30) == 1.0


@pytest.mark.parametrize("nbytes", [40, 60, 80, 100, 200, 400])
def test_48k_bitrates(nbytes):
    """LTPF on (low rates), lsb_mode (>= 1120 bits), nbits_ari 4 and 5 (> 1280, > 2560 bits)."""
    assert assert_encoder_parity(48000, 10, nbytes, 64, 40) == 1.0


def test_host_entry_point_and_ragged_counts():
    assert assert_encoder_parity(32000, 10, 80, 33, 12, host=True) == 1.0
    assert assert_encoder_parity(24000, 7.5, 45, 1, 12) == 1.0


def test_pipelined_host_entry_point():
    """lc3b_encoder_set_host_pipelining: the upload of call i+1 overlaps the kernels of call i; bytes are unchanged."""
    import torch

    import lc3_codec_b200 as L
    from common import corpus
    pcm, o_frames = corpus(48000, 10, 120, 70, 12)
    S, F, nf = pcm.shape
    sf, fd = L.SamplingFrequency.Hz48000, L.FrameDuration.TenMs
    ws = torch.empty(L.Lc3BatchEncoder.calc_working_buffer_lengths(S, fd, sf, 120), dtype=torch.uint8, device="cuda:0")
    enc = L.Lc3BatchEncoder(S, fd, sf, ws, 120)
    enc.set_host_pipelining(True)
    host_in = torch.from_numpy(np.ascontiguousarray(pcm.transpose(1, 0, 2))).pin_memory()          # [F,S,nf]
    host_out = torch.zeros((F, S, 120), dtype=torch.uint8).pin_memory()
    for f in range(F):
        enc.encode_frames_host(host_in[f], host_out[f])      # no synchronisation between calls
    torch.cuda.synchronize()
    assert np.array_equal(host_out.numpy().transpose(1, 0, 2), o_frames)


def test_odd_pcm_stride_and_unaligned_rows():
    """pcm_in rows at an odd sample pitch / 2-byte-aligned base take the kernels' one-sample load path; same bytes."""
    import torch

    import lc3_codec_b200 as L
    for fs, ms, nb in ((48000, 10, 120), (16000, 7.5, 30)):
        pcm, o_frames = corpus(fs, ms, nb, 40, 6)
        sf, fd = L.SamplingFrequency.from_hz(fs), L.FrameDuration.from_ms(ms)
        ws = torch.empty(L.Lc3BatchEncoder.calc_working_buffer_lengths(40, fd, sf, nb), dtype=torch.uint8, device="cuda:0")
        enc = L.Lc3BatchEncoder(40, fd, sf, ws, nb)
        nf = enc.nf
        backing = torch.zeros(40 * (nf + 3) + 1, dtype=torch.int16, device="cuda:0")
        view = backing[1:].view(40, nf + 3)[:, :nf]            # base 2-byte aligned only, pitch nf + 3 (odd)
        out = torch.zeros((40, nb), dtype=torch.uint8, device="cuda:0")
        for f in range(6):
            view.copy_(torch.from_numpy(np.ascontiguousarray(pcm[:, f])).cuda())
            enc.encode_frames(view, out)
            assert np.array_equal(out.cpu().numpy(), o_frames[:, f])


def test_8k_rejected_like_the_reference():
    """Lc3Encoder::new panics at 8 kHz (bandwidth_detector.rs:42-56) -> LC3B_ERR_INVALID_ARG."""
    import lc3_codec_b200 as L
    with pytest.raises(L.Lc3bError):
        L.Lc3BatchEncoder.calc_working_buffer_lengths(4, L.FrameDuration.TenMs, L.SamplingFrequency.Hz8000, 40)


def test_round_trip_gpu_encode_gpu_decode():
    """BASELINE config 5's shape at test size: GPU encode -> GPU decode equals oracle encode -> oracle decode (bit exact
    with the engine's inverse MDCT in the oracle, +-1 LSB with the reference's)."""
    from common import assert_pcm_matches_oracle, corpus, gpu_decode
    from oracle import pyoracle as O
    pcm, o_frames = corpus(48000, 10, 150, 64, 20)
    g_frames = gpu_encode(48000, 10, pcm, 150)
    g_pcm = gpu_decode(48000, 10, g_frames, trace=False)[0]
    assert_pcm_matches_oracle(g_pcm, 48000, 10, o_frames)


def test_sharded_encoder_and_graph_executor():
    """lc3b_sharded_encoder_* (two shards on device 0, host buffers for the whole batch) and lc3b_encoder_set_graph_mode:
    bytes identical to the oracle encoder either way."""
    import torch

    import lc3_codec_b200 as L
    pcm, o_frames = corpus(48000, 10, 120, 75, 10)
    S, F, nf = pcm.shape
    enc = L.Lc3ShardedBatchEncoder(S, L.FrameDuration.TenMs, L.SamplingFrequency.Hz48000, 120, devices=[0, 0])
    host_in = torch.from_numpy(np.ascontiguousarray(pcm.transpose(1, 0, 2))).pin_memory()
    host_out = torch.zeros((F, S, 120), dtype=torch.uint8).pin_memory()
    for f in range(F):
        enc.encode_frames_host(host_in[f], host_out[f])
    enc.wait()
    assert np.array_equal(host_out.numpy().transpose(1, 0, 2), o_frames)
    for graph in (True, False):
        sf, fd = L.SamplingFrequency.Hz48000, L.FrameDuration.TenMs
        ws = torch.empty(L.Lc3BatchEncoder.calc_working_buffer_lengths(S, fd, sf, 120), dtype=torch.uint8, device="cuda:0")
        e1 = L.Lc3BatchEncoder(S, fd, sf, ws, 120)
        e1.set_graph_mode(graph)
        out = torch.zeros((F, S, 120), dtype=torch.uint8, device="cuda:0")
        x = torch.from_numpy(np.ascontiguousarray(pcm.transpose(1, 0, 2))).cuda()
        for f in range(F):
            e1.encode_frames(x[f], out[f])
        assert np.array_equal(out.cpu().numpy().transpose(1, 0, 2), o_frames), graph


@pytest.mark.parametrize("fs,ms,nbytes", [(48000, 10, 150), (16000, 7.5, 30)])
def test_stage_level_parity_through_debug_read(fs, ms, nbytes):
    """lc3b_encoder_debug_read: the intermediates the kernels hand to each other, against the ORACLE'S STAGES chained by
    hand on the same frames (the stage functions the reference's own #[test]s pin: modified_dct_encode, attack_detector_run,
    long_term_post_filter_run, bandwidth_detector_run, sns_run, temporal_noise_shaping_run, spectral_quantization_run):
      e_b   band energies after the MDCT                      bit exact
      hand  near-Nyquist flag, attack flag, pitch index / present, LTPF active, LTPF bits
      xf    spectrum after SNS and TNS (the quantiser's input) bit exact
      xq    quantised spectrum                                 exact
    A byte-identical frame could in principle hide two compensating errors; these cannot."""
    import ctypes as C

    from oracle import pyoracle as O
    lib = O.lib()
    lib.lc3o_quant_new.restype = C.c_void_p
    sf, fd = O.SF[fs], O.FD[ms]
    cfg = O.config(fs, ms)
    nf, ne, fs_ind = cfg["nf"], cfg["ne"], cfg["fs_ind"]
    S, F = 6, 8
    pcm, _ = corpus(fs, ms, nbytes, S, F, first_stream=3)
    _, dbg = gpu_encode(fs, ms, pcm, nbytes, debug=True)
    nbits = nbytes * 8
    for s_ in range(S):
        mdct, att, ltpf = (C.c_void_p(getattr(lib, f"lc3o_{n}_new")(sf, fd)) for n in ("encmdct", "attack", "encltpf"))
        quant = C.c_void_p(lib.lc3o_quant_new(ne, fs_ind))
        for f in range(F):
            x16 = np.ascontiguousarray(pcm[s_, f])
            spec, eb = np.zeros(nf, np.float32), np.zeros(64, np.float32)
            near_nyquist = lib.lc3o_encmdct_run(mdct, O.p(x16), O.p(spec), O.p(eb))
            attack = lib.lc3o_attack_run(att, O.p(x16), nbytes)
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
            where = (fs, s_, f)
            assert np.array_equal(g_eb.view(np.uint32), eb.view(np.uint32)), where
            assert g_hand[:6].tolist() == [near_nyquist, attack, int(lt[0]), int(lt[1]), int(lt[2]), int(lt[3])], where
            assert np.array_equal(g_xf.view(np.uint32), spec[:ne].view(np.uint32)), where
            assert np.array_equal(g_xq, xq), where
        lib.lc3o_encmdct_free(mdct)
        lib.lc3o_attack_free(att)
        lib.lc3o_encltpf_free(ltpf)
        lib.lc3o_quant_free(quant)
