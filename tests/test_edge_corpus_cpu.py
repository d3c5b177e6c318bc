"""The edge material of tools/edge_corpus.py reaches the codec paths it exists for.  Oracle only (no GPU): the oracle's
own traces (LC3B_TRACE_* words of its decoder on its encoder's bitstreams) and its attack-detector stage."""
import ctypes as C
import functools

import numpy as np
import pytest

from oracle import pyoracle as O
from tools import edge_corpus as E
from tools.corpus import MIXED_NBYTES

ALL_CONFIGS = sorted(MIXED_NBYTES)
TR = O.TR
N_CLS = len(E.CLASSES)


@functools.lru_cache(maxsize=16)
def _run(fs, ms, nbytes, n_var=4, n_frames=6):
    """Every class in n_var variants through the oracle: (pcm, frames, decoded pcm, trace)."""
    pcm = E.make_edge_pcm(N_CLS * n_var, n_frames, fs, ms)
    frames = O.encode_streams(pcm, fs, ms, nbytes)
    dec, tr, _, _ = O.decode_streams(frames, fs, ms, trace=True)
    return pcm, frames, dec, tr


def _cls(tr, name):
    return tr[[s for s in range(tr.shape[0]) if E.edge_class(s) == name]]


@pytest.mark.parametrize("fs,ms", ALL_CONFIGS)
def test_shapes_and_counter_based(fs, ms):
    nf = O.config(fs, ms)["nf"]
    assert E.frame_geometry(fs, ms) == (nf, O.config(fs, ms)["z"])
    a = E.make_edge_pcm(2 * N_CLS, 3, fs, ms)
    assert a.shape == (2 * N_CLS, 3, nf) and a.dtype == np.int16
    assert np.array_equal(E.make_edge_pcm(5, 3, fs, ms, first_stream=7), a[7:12])
    assert np.array_equal(E.make_edge_streams([3, 20], 3, fs, ms), a[[3, 20]])


@pytest.mark.parametrize("fs,ms,nbytes", [(48000, 10, 20), (48000, 10, 400), (44100, 10, 20), (44100, 10, 400),
                                          (48000, 7.5, 20)])
def test_global_gain_reaches_both_clamps(fs, ms, nbytes):
    """Full-scale noise puts gg_ind on its clamp of 255 in every frame (the quantiser's gg_ind < 255 branch and its
    gain floor from xmax); digital silence gives 0 (xmax == 0)."""
    _, _, _, tr = _run(fs, ms, nbytes)
    assert (_cls(tr, "noise_fs")[..., TR["GG_IND"]] == 255).all()
    assert (_cls(tr, "silence")[..., TR["GG_IND"]] == 0).all()


@pytest.mark.parametrize("fs,ms,nbytes", [(48000, 10, 20), (48000, 10, 400), (16000, 7.5, 20), (8000, 10, 20)])
def test_decoded_pcm_saturates_both_ways(fs, ms, nbytes):
    _, _, dec, _ = _run(fs, ms, nbytes)
    assert (dec == 32767).any() and (dec == -32768).any()


def test_lsb_mode_and_zero_frames():
    _, _, _, tr = _run(48000, 10, 400)
    assert (_cls(tr, "noise_fs")[..., TR["LSB_MODE"]] == 1).all()
    assert (_cls(tr, "silence")[..., TR["IS_ZERO"]] == 1).all()
    _, _, _, tr = _run(16000, 7.5, 20)
    assert (_cls(tr, "silence")[..., TR["IS_ZERO"]] == 1).all()


@pytest.mark.parametrize("fs,ms", ALL_CONFIGS)
def test_every_bandwidth_index(fs, ms):
    """The low-passed noise and the tones make the bandwidth detector signal every index the configuration can.  At
    44.1 / 48 kHz and 10 ms that excludes 3 (super wideband): its cutoff test reads the bands start - l + 1 .. start - 1
    with l = 1, an empty range, so the detector falls through to full band (bandwidth_detector.rs)."""
    fs_ind = O.config(fs, ms)["fs_ind"]
    _, _, _, tr = _run(fs, ms, 60)
    can = set(range(fs_ind + 1)) - ({3} if fs_ind == 4 and ms == 10 else set())
    assert set(np.unique(tr[..., TR["BW"]]).tolist()) == can


@pytest.mark.parametrize("fs,ms", [(48000, 10), (48000, 7.5), (32000, 10), (32000, 7.5)])
def test_two_tns_filters(fs, ms):
    _, _, _, tr = _run(fs, ms, 120)
    assert (tr[..., TR["NUM_TNS"]] == 2).any()
    assert (_cls(tr, "step")[..., TR["RC_ORDER0"]] > 0).any()


@pytest.mark.parametrize("fs,ms,nbytes", [(32000, 10, 81), (32000, 7.5, 61), (32000, 7.5, 149), (48000, 10, 100),
                                          (48000, 10, 400), (44100, 7.5, 75), (48000, 7.5, 149)])
def test_attack_flag_is_set(fs, ms, nbytes):
    """The oracle's attack detector (attack_detector.rs) flags the steps and impulses wherever it is active."""
    lib = O.lib()
    pcm = E.make_edge_streams(E.streams_of("step", 2) + E.streams_of("impulse", 3), 6, fs, ms)
    flags = np.zeros(pcm.shape[:2], bool)
    for s in range(pcm.shape[0]):
        att = C.c_void_p(lib.lc3o_attack_new(O.SF[fs], O.FD[ms]))
        for f in range(pcm.shape[1]):
            flags[s, f] = lib.lc3o_attack_run(att, O.p(np.ascontiguousarray(pcm[s, f])), nbytes)
        lib.lc3o_attack_free(att)
    assert flags[:2].any(-1).all(), "every step is an attack"
    assert flags[2:].any()


@pytest.mark.parametrize("fs,ms,nbytes", [(48000, 10, 20), (48000, 7.5, 30), (16000, 7.5, 20), (32000, 10, 40),
                                          (24000, 10, 30)])
def test_ltpf_active_at_both_ends_of_the_pitch_range(fs, ms, nbytes):
    _, _, _, tr = _run(fs, ms, nbytes)
    t = _cls(tr, "pulses")
    pi = t[..., TR["PITCH_INDEX"]][t[..., TR["LTPF_ACTIVE"]] == 1]
    assert pi.size and pi.min() <= 16 and pi.max() >= 500, np.unique(pi)


@pytest.mark.parametrize("fs,ms", [(16000, 7.5), (48000, 10), (44100, 7.5)])
def test_edge_material_spans_the_gain_range(fs, ms):
    """Beyond the clamps: the classes spread gg_ind over much of its range at one rate."""
    _, _, _, tr = _run(fs, ms, 100)
    gg = np.unique(tr[..., TR["GG_IND"]])
    assert gg.min() == 0 and gg.max() >= 240 and gg.size >= 40


def test_rate_boundaries_follow_the_reference_formulas():
    """Spot values of the restated thresholds, and the 7.5 ms rounding: 32 * nbytes / 3 is an integer or a third
    away from one, never within half a bit below an even threshold, so round() and truncation put every gain row and the
    post filter's end at the same frame length."""
    assert E.rate_boundaries(4, 48000, 10)["rate_flag"] == [101]       # 100 B is the last length below the switch
    assert E.rate_boundaries(1, 16000, 10)["gg_off"] == [288]          # the offset saturates at 288 B at 16 kHz
    assert E.rate_boundaries(4, 48000, 7.5)["attack"] == [75, 150]
    assert E.ltpf_impossible_from(4, 10) == 110 and E.ltpf_impossible_from(1, 7.5) == 60
    for fs_ind in range(5):
        for thr in (320, 400, 480, 560):
            for b in range(1, 401):
                nb = 8 * b
                assert (E.t_nbits(b, 7.5) >= thr + 80 * fs_ind) == (int(nb * 10.0 / 7.5) >= thr + 80 * fs_ind)
    for fs, ms in ALL_CONFIGS:
        for b in E.boundary_lengths(O.config(fs, ms)["fs_ind"], fs, ms):
            assert E.MIN_NBYTES <= b <= E.MAX_NBYTES
