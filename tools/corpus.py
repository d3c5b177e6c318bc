"""Deterministic synthetic audio corpus (SURVEY.md section 8d) for parity tests and bench.py.

Stream `s` draws every parameter from splitmix64(0x4C43330000000000 + s); its signal class is
`s mod 3`:
  0  log sine sweep 50 Hz -> 0.45*fs over the clip, amplitude 0.1..0.9 FS
  1  Gaussian noise, -40..-6 dBFS, one-pole spectral tilt, two 100 ms silent gaps
     (exercises zero frames, low gains, the bandwidth detector)
  2  speech-like: harmonic stack f0 in [90,260] Hz with 5 Hz +-3 % vibrato, 3..6 Hz syllabic AM,
     three formant-weighted harmonic groups, voiced/unvoiced alternation every 150..400 ms
     (exercises LTPF on/off/pitch-change transitions, TNS, attacks)
Everything is vectorised numpy, counter-based (no sequential RNG state), so any sub-range of
streams can be generated independently and identically on any machine.

This is bench/test data, not part of the codec path.
"""
from __future__ import annotations

from pathlib import Path

import numpy as np
from scipy.signal import lfilter

SEED0 = np.uint64(0x4C43330000000000)
GOLD = np.uint64(0x9E3779B97F4A7C15)
TILT_POLES = np.array([-0.6, -0.3, 0.0, 0.3, 0.5, 0.7, 0.8, 0.9])


def _mix(z: np.ndarray) -> np.ndarray:
    with np.errstate(over="ignore"):
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def _draw(seed: np.ndarray, k: int) -> np.ndarray:
    """k-th uniform [0,1) draw of each stream's splitmix64 sequence."""
    with np.errstate(over="ignore"):
        st = seed + GOLD * np.uint64(k + 1)
    return (_mix(st) >> np.uint64(11)).astype(np.float64) * (1.0 / (1 << 53))


def _noise(seed: np.ndarray, n: int, lane: int) -> np.ndarray:
    """[streams, n] standard normal, counter-based (Box-Muller on two hashed uniforms)."""
    with np.errstate(over="ignore"):
        base = _mix(seed + GOLD * np.uint64(1000 + lane))[:, None]
        ctr = np.arange(n, dtype=np.uint64)[None, :]
        u1 = (_mix(base + GOLD * (ctr * np.uint64(2))) >> np.uint64(11)).astype(np.float64) * (1.0 / (1 << 53))
        u2 = (_mix(base + GOLD * (ctr * np.uint64(2) + np.uint64(1))) >> np.uint64(11)).astype(np.float64) * (1.0 / (1 << 53))
    return (np.sqrt(-2.0 * np.log(1.0 - u1)) * np.cos(2.0 * np.pi * u2)).astype(np.float32)


def _sweep(seed, fs, n):
    t = np.arange(n, dtype=np.float64) / fs
    T = n / fs
    f0, f1 = 50.0, 0.45 * fs
    k = f1 / f0
    phase = 2.0 * np.pi * f0 * T / np.log(k) * (np.power(k, t / T) - 1.0)
    amp = 0.1 + 0.8 * _draw(seed, 0)
    ph0 = 2.0 * np.pi * _draw(seed, 1)
    return (amp[:, None] * np.sin(phase[None, :] + ph0[:, None])).astype(np.float32)


def _tilted_noise(seed, fs, n):
    level_db = -40.0 + 34.0 * _draw(seed, 0)
    rms = np.power(10.0, level_db / 20.0)
    pole_idx = np.minimum((_draw(seed, 1) * len(TILT_POLES)).astype(int), len(TILT_POLES) - 1)
    x = _noise(seed, n, 0)
    out = np.empty_like(x)
    for pi, a in enumerate(TILT_POLES):
        sel = np.nonzero(pole_idx == pi)[0]
        if sel.size:
            y = lfilter([np.sqrt(1.0 - a * a)], [1.0, -a], x[sel].astype(np.float64), axis=1)
            out[sel] = y.astype(np.float32)
    out *= rms[:, None].astype(np.float32)
    gap = int(0.1 * fs)
    idx = np.arange(n)[None, :]
    for g in (2, 3):
        start = (_draw(seed, g) * max(1, n - gap)).astype(int)[:, None]
        out[(idx >= start) & (idx < start + gap)] = 0.0
    return out


def _speech(seed, fs, n):
    t = np.arange(n, dtype=np.float64)[None, :] / fs
    f0 = (90.0 + 170.0 * _draw(seed, 0))[:, None]
    vib_ph = (2 * np.pi * _draw(seed, 1))[:, None]
    # phase = 2*pi*integral f0*(1+0.03 sin(2 pi 5 t)) dt
    phase = 2 * np.pi * f0 * (t - 0.03 / (2 * np.pi * 5.0) * (np.cos(2 * np.pi * 5.0 * t + vib_ph) - np.cos(vib_ph)))
    am_f = (3.0 + 3.0 * _draw(seed, 2))[:, None]
    env = 0.55 + 0.45 * np.sin(2 * np.pi * am_f * t + (2 * np.pi * _draw(seed, 3))[:, None])
    formants = np.stack([500 + 300 * _draw(seed, 4), 1200 + 1000 * _draw(seed, 5), 2500 + 800 * _draw(seed, 6)], 1)
    bws = np.array([120.0, 180.0, 250.0])
    fmax = min(0.45 * fs, 5000.0)
    hmax = int(fmax // 90.0)
    # Chebyshev recurrence for sin(h*phase): s_h = 2 cos(p) s_{h-1} - s_{h-2}
    c = np.cos(phase).astype(np.float32)
    s1 = np.sin(phase).astype(np.float32)
    s_prev, s_cur = np.zeros_like(s1), s1
    voiced = np.zeros_like(s1)
    for h in range(1, hmax + 1):
        fh = h * f0[:, 0]
        w = np.zeros_like(fh)
        for j in range(3):
            w += 1.0 / (1.0 + ((fh - formants[:, j]) / bws[j]) ** 2)
        w = np.where(fh < fmax, w + 0.02, 0.0) / h ** 0.5
        voiced += (w.astype(np.float32))[:, None] * s_cur
        s_prev, s_cur = s_cur, 2.0 * c * s_cur - s_prev
    voiced *= (0.25 * env).astype(np.float32)
    # unvoiced: differentiated (high-passed) noise bursts
    nz = _noise(seed, n, 1)
    unv = np.empty_like(nz)
    unv[:, 0] = nz[:, 0]
    unv[:, 1:] = nz[:, 1:] - nz[:, :-1]
    unv *= (0.04 * env).astype(np.float32)
    # voiced/unvoiced alternation: segment lengths 150..400 ms from per-stream draws
    seg_id = np.zeros((seed.shape[0], n), dtype=np.int32)
    pos = np.zeros(seed.shape[0], dtype=np.int64)
    idx = np.arange(n)[None, :]
    k = 0
    while (pos < n).any() and k < 64:
        ln = ((0.15 + 0.25 * _draw(seed, 10 + k)) * fs).astype(np.int64)
        seg_id[(idx >= pos[:, None]) & (idx < (pos + ln)[:, None])] = k
        pos += ln
        k += 1
    is_voiced = (seg_id % 3) != 2                    # two voiced segments, one unvoiced
    amp = (0.3 + 0.6 * _draw(seed, 7))[:, None].astype(np.float32)
    return amp * np.where(is_voiced, voiced, unv)


def make_pcm(n_streams: int, n_frames: int, fs: int, nf: int, first_stream: int = 0) -> np.ndarray:
    """[n_streams, n_frames, nf] int16.  fs is the nominal rate (44100 uses nf of 48 kHz, like the reference)."""
    n = n_frames * nf
    ids = np.arange(first_stream, first_stream + n_streams, dtype=np.uint64)
    with np.errstate(over="ignore"):
        seed = SEED0 + ids
    out = np.zeros((n_streams, n), dtype=np.float32)
    cls = (ids % np.uint64(3)).astype(int)
    for c, fn in ((0, _sweep), (1, _tilted_noise), (2, _speech)):
        sel = np.nonzero(cls == c)[0]
        for i in range(0, sel.size, 512):             # bound temporary memory
            chunk = sel[i:i + 512]
            out[chunk] = fn(seed[chunk], float(fs), n)
    x = out.astype(np.float64) * 32768.0
    q = np.where(x >= 0, np.floor(x + 0.5), np.ceil(x - 0.5))   # round half away from zero
    return np.clip(q, -32768, 32767).astype(np.int16).reshape(n_streams, n_frames, nf)


# nbytes used by the mixed-rate config (SURVEY.md 8d): (fs, ms) -> nbytes
MIXED_NBYTES = {(8000, 7.5): 20, (8000, 10): 26, (16000, 7.5): 30, (16000, 10): 40, (24000, 7.5): 45, (24000, 10): 60,
                (32000, 7.5): 60, (32000, 10): 80, (44100, 7.5): 90, (44100, 10): 120, (48000, 7.5): 90, (48000, 10): 120}


# ---- SURVEY.md 8d clips: 200 frames per stream; benches and full-size tests take a window of consecutive frames
CLIP_FRAMES, CLIP_SKIP = 200, 10


def clip_offsets(n_streams: int, n_frames: int, first_stream: int = 0) -> np.ndarray:
    """Per-stream first frame of an n_frames window inside the 200-frame clip, in [CLIP_SKIP, CLIP_FRAMES - n_frames]
    (draw 40 of the stream's splitmix64 sequence): the windows of a batch sample the whole clip."""
    ids = np.arange(first_stream, first_stream + n_streams, dtype=np.uint64)
    with np.errstate(over="ignore"):
        u = _draw(SEED0 + ids, 40)
    span = CLIP_FRAMES - n_frames - CLIP_SKIP
    return CLIP_SKIP + np.minimum((u * (span + 1)).astype(int), span)


def take_window(clips: np.ndarray, off: np.ndarray, n_frames: int, lead: int = 0) -> np.ndarray:
    """[S, CLIP_FRAMES, ...] -> [S, lead + n_frames, ...]: frames off-lead .. off+n_frames-1 of every stream."""
    idx = (off - lead)[:, None] + np.arange(lead + n_frames)[None, :]
    return np.ascontiguousarray(clips[np.arange(clips.shape[0])[:, None], idx])


def make_pcm_window(n_streams: int, n_frames: int, fs: int, nf: int, lead: int = 0, first_stream: int = 0) -> np.ndarray:
    """[n_streams, lead + n_frames, nf] int16 cut from the streams' 200-frame clips at clip_offsets(); `lead` extra
    frames in front of the window let an encoder settle before the frames that count (lead <= CLIP_SKIP)."""
    assert 0 <= lead <= CLIP_SKIP
    out = np.empty((n_streams, lead + n_frames, nf), np.int16)
    for i in range(0, n_streams, 256):                    # bound temporary memory
        n = min(256, n_streams - i)
        clips = make_pcm(n, CLIP_FRAMES, fs, nf, first_stream + i)
        out[i:i + n] = take_window(clips, clip_offsets(n, n_frames, first_stream + i), n_frames, lead)
    return out


# ---- the 48 kHz / 10 ms / 150 B bench fixture of tools/make_bench_corpus.py, [1024, 8, 150] u8: stored as two halves of
# 512 streams so that every golden file stays under 1 MB
GOLDEN = Path(__file__).resolve().parent.parent / "tests" / "golden"
BENCH_C1_PARTS = ("bench_c1_frames_0.npy", "bench_c1_frames_1.npy")


def load_bench_c1_frames() -> np.ndarray:
    return np.concatenate([np.load(GOLDEN / p) for p in BENCH_C1_PARTS])
