"""Deterministic edge-of-range test signals: the inputs the synthetic corpus of tools/corpus.py never produces on purpose.

Stream `s` belongs to class `s mod len(CLASSES)` and to variant `s // len(CLASSES)` of that class; every random draw is
counter-based (splitmix64 of a per-stream seed, like tools/corpus.py), so any sub-range of streams can be generated on
its own and comes out identical on every machine.

  silence      digital silence                                        gg_ind 0, zero frames
  dither       +-1 LSB uniform dither
  dc_pos       DC at +32767
  dc_neg       DC at -32768
  noise_fs     full-scale uniform white noise (every int16 value)     gg_ind 255, the xmax gain floor, lsb_mode, clipping
  square       full-scale square wave, period 6 / 40 / 250 samples    clipped decoder output
  nyquist      alternating +32767 / -32768
  impulse      one full-scale impulse in frame 1, at sample 0, at nf - 1, or nf - z/2 (inside the window's zero tail,
               which this frame's transform skips and the next frame's sees)
  step         silence, then from the middle of frame 1 on: DC at +32767, or full-scale noise (attacks, two TNS filters
               where the bandwidth has them)
  tone         0.7 FS sine at 0.49 fs, or 1 kHz below / 250 Hz above one of the bandwidth detector's cutoffs (4, 8, 12,
               16 kHz)
  lowpass      white noise brick-walled at 0.85 x one of the cutoffs (the detector's lower bandwidth indices: a tone's
               window leakage keeps the bands above it too loud at 48 kHz)
  pulses       full-scale pulse train at the LTPF's shortest / longest pitch lag (32 / 228 samples at 12.8 kHz), at lag 36
               (32 and 33 lie below the open-loop search's 17 samples at 6.4 kHz and come out as their octave; 36 is the
               shortest lag that is found as itself at every configuration), or lag 36 jumping to 228 half way through
  gap_noise    1..3 silent frames, then loud uniform noise

This is test data, not part of the codec path.
"""
from __future__ import annotations

import numpy as np

from tools.corpus import GOLD, _draw, _mix

SEED_EDGE = np.uint64(0x4C43334544474500)
CLASSES = ("silence", "dither", "dc_pos", "dc_neg", "noise_fs", "square", "nyquist", "impulse", "step", "tone", "lowpass",
           "pulses", "gap_noise")
SQUARE_PERIODS = (6, 40, 250)
BW_CUTOFFS_HZ = (4000, 8000, 12000, 16000)
LTPF_LAGS_12K8 = (32, 36, 228)


def edge_class(stream: int) -> str:
    return CLASSES[stream % len(CLASSES)]


def streams_of(cls: str, n: int, first: int = 0) -> list[int]:
    """The first n stream ids >= first whose class is `cls` (its variants in order)."""
    c = CLASSES.index(cls)
    s0 = first + (c - first) % len(CLASSES)
    return [s0 + k * len(CLASSES) for k in range(n)]


def tone_freqs(fs: int) -> list[float]:
    """The tone class's frequencies at fs: 0.49 fs, then either side of every cutoff below fs / 2."""
    out = [0.49 * fs]
    for c in BW_CUTOFFS_HZ:
        if c + 250 < fs / 2:
            out += [c - 1000.0, c + 250.0]
    return out


def _uniform16(seed: int, n: int) -> np.ndarray:
    """n uniform int16 values (all 65536 equally likely), counter-based."""
    with np.errstate(over="ignore"):
        base = _mix(np.uint64(seed) + GOLD * np.uint64(777))
        ctr = np.arange(n, dtype=np.uint64)
        return (_mix(base + GOLD * ctr) >> np.uint64(48)).astype(np.uint16).view(np.int16)


def _pulse_period(lag12k8: int, fs: int) -> float:
    """Pitch lag at 12.8 kHz -> samples at fs (44.1 kHz runs the LTPF as if it were 48 kHz, like the reference)."""
    return lag12k8 * (8000.0 * np.ceil(fs / 8000.0)) / 12800.0


def _pulse_train(period: float, n: int, start: int = 0) -> np.ndarray:
    x = np.zeros(n, np.int32)
    pos = np.arange(start, n, period)
    x[np.floor(pos).astype(int)] = 32767
    return x


def frame_geometry(fs: int, ms: float) -> tuple[int, int]:
    """(nf, z): samples per frame (44.1 kHz frames hold as many as 48 kHz ones) and the length of the analysis
    window's zero tail."""
    nf = int(round((48000 if fs == 44100 else fs) * ms / 1000.0))
    return nf, (3 * nf // 8 if ms == 10 else 7 * nf // 30)


def _stream(sid: int, n_frames: int, fs: int, ms: float) -> np.ndarray:
    nf, z = frame_geometry(fs, ms)
    n = n_frames * nf
    cls = edge_class(sid)
    var = sid // len(CLASSES)
    with np.errstate(over="ignore"):
        seed = int(SEED_EDGE + np.uint64(sid))
    t = np.arange(n)
    if cls == "silence":
        return np.zeros(n, np.int32)
    if cls == "dither":
        return (_uniform16(seed, n).astype(np.int32) % 3) - 1
    if cls == "dc_pos":
        return np.full(n, 32767, np.int32)
    if cls == "dc_neg":
        return np.full(n, -32768, np.int32)
    if cls == "noise_fs":
        return _uniform16(seed, n).astype(np.int32)
    if cls == "square":
        per = SQUARE_PERIODS[var % len(SQUARE_PERIODS)]
        return np.where((t % per) < per // 2, 32767, -32768)
    if cls == "nyquist":
        return np.where(t % 2 == 0, 32767, -32768)
    if cls == "impulse":
        pos = (0, nf - 1, nf - z // 2)[var % 3]
        x = np.zeros(n, np.int32)
        x[min(1, n_frames - 1) * nf + pos] = 32767
        return x
    if cls == "step":
        on = min(1, n_frames - 1) * nf + nf // 2
        x = np.full(n, 32767, np.int32) if var % 2 == 0 else _uniform16(seed, n).astype(np.int32)
        x[:on] = 0
        return x
    if cls == "tone":
        freqs = tone_freqs(fs)
        f = freqs[var % len(freqs)]
        ph = 2 * np.pi * _draw(np.array([np.uint64(seed)]), 0)[0]
        return np.round(0.7 * 32767.0 * np.sin(2 * np.pi * f / fs * t + ph)).astype(np.int32)
    if cls == "lowpass":
        cuts = [c for c in BW_CUTOFFS_HZ if c < fs / 2] or [fs / 2]
        spec = np.fft.rfft(_uniform16(seed, n).astype(np.float64))
        spec[np.fft.rfftfreq(n, 1.0 / fs) > 0.85 * cuts[var % len(cuts)]] = 0.0
        x = np.fft.irfft(spec, n)
        return np.round(x * (0.5 * 32767.0 / max(np.abs(x).max(), 1.0))).astype(np.int32)
    if cls == "pulses":
        v = var % 4
        if v < 3:
            return _pulse_train(_pulse_period(LTPF_LAGS_12K8[v], fs), n)
        half = (n_frames // 2) * nf
        x = _pulse_train(_pulse_period(LTPF_LAGS_12K8[1], fs), n)
        x[half:] = _pulse_train(_pulse_period(LTPF_LAGS_12K8[2], fs), n - half)
        return x
    if cls == "gap_noise":
        k = 1 + var % 3
        x = (_uniform16(seed, n).astype(np.int32) * 3) // 4
        x[:k * nf] = 0
        return x
    raise AssertionError(cls)


def make_edge_streams(ids, n_frames: int, fs: int, ms: float) -> np.ndarray:
    """[len(ids), n_frames, nf] int16: the edge streams with the given ids."""
    nf = frame_geometry(fs, ms)[0]
    out = np.empty((len(ids), n_frames * nf), np.int16)
    for i, sid in enumerate(ids):
        out[i] = np.clip(_stream(int(sid), n_frames, fs, ms), -32768, 32767)
    return out.reshape(len(ids), n_frames, nf)


def make_edge_pcm(n_streams: int, n_frames: int, fs: int, ms: float, first_stream: int = 0) -> np.ndarray:
    """[n_streams, n_frames, nf] int16 edge material; stream i is edge stream first_stream + i."""
    return make_edge_streams(range(first_stream, first_stream + n_streams), n_frames, fs, ms)


# ---- the reference's integer rate decisions, restated from its formulas (not from the engine) so that tests can put
# frame lengths on either side of each.  fs_ind: 0..4 for 8 / 16 / 24 / 32 / 44.1 and 48 kHz.
MIN_NBYTES, MAX_NBYTES = 20, 400


def t_nbits(nbytes: int, ms: float) -> int:
    """The LTPF's 10 ms-equivalent frame bits: round(nbits * 10 / 7.5) at 7.5 ms (Rust's f64::round, half away from
    zero; 32 * nbytes / 3 is never a half, so Python's round() agrees)."""
    nbits = 8 * nbytes
    return int(round(nbits * 10.0 / 7.5)) if ms == 7.5 else nbits


def _first(pred) -> int | None:
    """First nbytes in [1, 400] where pred turns true (pred is monotone in nbytes), None if it never does."""
    return next((b for b in range(1, MAX_NBYTES + 1) if pred(b)), None)


def rate_boundaries(fs_ind: int, fs: int, ms: float) -> dict[str, list[int]]:
    """name -> the frame lengths b at which a decision changes between b - 1 and b:
      rate_flag     arithmetic-coder context switch, nbits > 160 + 160 fs_ind
      lsb_mode      LSB mode allowed, nbits >= 480 + 160 fs_ind
      nbits_ari     nbits <= 1280 / <= 2560
      gg_off        global-gain offset min(115, nbits / (10 (fs_ind + 1))) saturates
      tns_lpc       TNS LPC weighting off: nbits >= 480 (10 ms) / >= 360 (7.5 ms)
      attack        attack detector switched on / off
      ltpf_gain     encoder gain_ltpf_on ends: t_nbits >= 560 + 80 fs_ind; the same length is the first at which the
                    decoder's post filter is impossible (gain row (0.0, 0))
      ltpf_rows     decoder post-filter gain rows: t_nbits >= 320 / 400 / 480 + 80 fs_ind"""
    sf = 80 * fs_ind
    out = {
        "rate_flag": [_first(lambda b: 8 * b > 160 + 160 * fs_ind)],
        "lsb_mode": [_first(lambda b: 8 * b >= 480 + 160 * fs_ind)],
        "nbits_ari": [_first(lambda b: 8 * b > 1280), _first(lambda b: 8 * b > 2560)],
        "gg_off": [_first(lambda b: (8 * b) // (10 * (fs_ind + 1)) >= 115)],
        "tns_lpc": [_first(lambda b: 8 * b >= (480 if ms == 10 else 360))],
        "ltpf_gain": [_first(lambda b: t_nbits(b, ms) >= 560 + sf)],
        "ltpf_rows": [_first(lambda b, r=r: t_nbits(b, ms) >= r + sf) for r in (320, 400, 480)],
    }
    if fs == 32000:
        out["attack"] = [81] if ms == 10 else [61, 150]
    elif fs >= 44100:
        out["attack"] = [100] if ms == 10 else [75, 150]
    return {k: sorted(b for b in v if b is not None) for k, v in out.items()}


def ltpf_impossible_from(fs_ind: int, ms: float) -> int:
    """The reference's first frame length from which the post filter can never act (gain row (0.0, 0))."""
    return _first(lambda b: t_nbits(b, ms) >= 560 + 80 * fs_ind)


def boundary_lengths(fs_ind: int, fs: int, ms: float) -> list[int]:
    """Every boundary b at b - 1, b and b + 1, plus 20, 21, 399 and 400, limited to [20, 400]."""
    s = {MIN_NBYTES, MIN_NBYTES + 1, MAX_NBYTES - 1, MAX_NBYTES}
    for bs in rate_boundaries(fs_ind, fs, ms).values():
        for b in bs:
            s.update(x for x in (b - 1, b, b + 1) if MIN_NBYTES <= x <= MAX_NBYTES)
    return sorted(s)
