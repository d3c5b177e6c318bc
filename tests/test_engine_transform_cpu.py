"""The engine's inverse MDCT as the oracle restates it (oracle/lc3o_engine_imdct.cpp), on the CPU.

The decoder's GPU PCM is compared bit for bit with the oracle run with this transform (transform="engine"), and within
+-1 LSB with the oracle run with the reference's (kissfft).  These tests are what make both gates meaningful:
- both DCT-IVs against a float64 DCT-IV at all nine sizes: the engine's is as accurate as kissfft, so keeping the
  +-1 LSB contract against the reference is justified (numbers in DESIGN.md section 2);
- the unfold, the folded window and the overlap-add against a float64 restatement of modified_dct.rs:97-151;
- the twiddle tables narrow to the same f32 values on any host or device whose f64 cos / sin are within 4 ulp;
- the engine mode changes nothing but the transform: same traces and spectra, PCM within +-1 LSB.
"""
import math

import numpy as np
import pytest
import scipy.fft

from common import corpus
from oracle import pyoracle as O
from tools.corpus import MIXED_NBYTES

# one configuration per DCT-IV size nf (the FFT is nf / 2 points)
NF_CONFIG = {60: (8000, 7.5), 80: (8000, 10), 120: (16000, 7.5), 160: (16000, 10), 180: (24000, 7.5), 240: (24000, 10),
             320: (32000, 10), 360: (48000, 7.5), 480: (48000, 10)}
# every distinct (nf, z, window) geometry of the unfold: 44.1 kHz shares 48 kHz's
GEOMETRIES = [(8000, 7.5), (8000, 10), (16000, 7.5), (16000, 10), (24000, 7.5), (24000, 10), (32000, 7.5), (32000, 10),
              (48000, 7.5), (48000, 10)]
# worst |y - y64| / (||x||_2 2^-24) over the inputs below, measured at 28.3 (engine, nf 480) and 25.7 (kissfft, nf 480)
ERR_BOUND = 48.0
# the engine's worst error over kissfft's at the same size, measured at most 1.23 (nf 160)
ENGINE_OVER_KISSFFT = 1.5


def _sf_fd(fs, ms):
    return O.SF[fs], O.FD[ms]


def _dct_iv_ref(x):
    """float64 DCT-IV in the scale of dct_iv.rs: y[k] = 2 sum_n x[n] cos(pi / nf (n + 1/2)(k + 1/2))."""
    return scipy.fft.dct(np.asarray(x, np.float64), type=4)


def _kissfft(x):
    y = np.ascontiguousarray(x, np.float32).copy()
    O.lib().lc3o_dct_iv(len(y), O.p(y))
    return y


def _engine(x, fs, ms):
    y = np.ascontiguousarray(x, np.float32).copy()
    O.lib().lc3o_engine_dct_iv(*_sf_fd(fs, ms), O.p(y))
    return y


def _corpus_spectra(fs, ms, nf):
    """Shaped spectra the oracle hands its inverse MDCT on corpus streams, zero padded to nf."""
    _, frames = corpus(fs, ms, MIXED_NBYTES[(fs, ms)], 16, 12)
    sp = O.decode_streams(frames, fs, ms, trace=True)[3]
    sp = sp.reshape(-1, sp.shape[-1])
    out = np.zeros((sp.shape[0], nf), np.float32)
    out[:, :sp.shape[1]] = sp
    return out[np.abs(out).sum(1) > 0]


def _inputs(nf, fs, ms):
    rng = np.random.default_rng(nf)
    return {"gaussian": rng.standard_normal((64, nf)).astype(np.float32),
            "uniform full scale": rng.uniform(-32768.0, 32768.0, (64, nf)).astype(np.float32),
            "impulse at every index": 32767.0 * np.eye(nf, dtype=np.float32),
            "corpus spectra": _corpus_spectra(fs, ms, nf)}


def test_kissfft_dct_iv_has_the_scale_of_the_float64_reference():
    """lc3o_dct_iv (the reference's transform) and scipy's unnormalised DCT-IV agree in scale: the float64 reference
    below needs no factor."""
    for nf in NF_CONFIG:
        x = np.random.default_rng(1).standard_normal(nf).astype(np.float32)
        r = _dct_iv_ref(x)
        assert abs(float(_kissfft(x).astype(np.float64) @ r / (r @ r)) - 1.0) < 1e-6, nf


@pytest.mark.parametrize("nf", sorted(NF_CONFIG))
def test_dct_iv_against_float64(nf):
    """Both f32 DCT-IVs against float64 on Gaussian, uniform full-scale, unit-impulse and corpus inputs: the worst error
    over ||x||_2 2^-24 is below ERR_BOUND for each, and the engine's is at most ENGINE_OVER_KISSFFT times kissfft's."""
    fs, ms = NF_CONFIG[nf]
    worst = {"kissfft": 0.0, "engine": 0.0}
    for kind, xs in _inputs(nf, fs, ms).items():
        assert len(xs) > 0, kind
        for x in xs:
            r = _dct_iv_ref(x)
            unit = float(np.linalg.norm(x.astype(np.float64))) * 2.0 ** -24
            for name, y in (("kissfft", _kissfft(x)), ("engine", _engine(x, fs, ms))):
                worst[name] = max(worst[name], float(np.abs(y.astype(np.float64) - r).max()) / unit)
    print(f"nf {nf}: worst error / (||x|| 2^-24): kissfft {worst['kissfft']:.2f}, engine {worst['engine']:.2f}")
    assert worst["kissfft"] < ERR_BOUND and worst["engine"] < ERR_BOUND, worst
    assert worst["engine"] <= ENGINE_OVER_KISSFFT * worst["kissfft"], worst


def test_engine_dct_iv_is_not_kissfft():
    """The two factorisations really differ (otherwise the exact gate would not need an engine mode)."""
    x = np.random.default_rng(2).standard_normal(480).astype(np.float32)
    assert not np.array_equal(_engine(x, 48000, 10), _kissfft(x))


def _tables(fs, ms):
    nf = O.config(fs, ms)["nf"]
    win, w = np.zeros(2 * nf, np.float32), np.zeros(2 * nf, np.float32)
    dtw, ftw = np.zeros((nf // 2, 2), np.float32), np.zeros((nf // 2, 2), np.float32)
    O.lib().lc3o_engine_tables(*_sf_fd(fs, ms), O.p(win), O.p(dtw), O.p(ftw))
    O.lib().lc3o_mdct_window(*_sf_fd(fs, ms), O.p(w))
    return win, w, dtw, ftw


def _unfold64(D, nf, z, w):
    """modified_dct.rs:97-136 in float64: t = [y, -rev(y)] rotated left by nf / 2, the wrapped quarter negated, times
    1 / sqrt(2 nf), times w[2 nf - 1 - n].  Returns (head, tail) = (t[z:z + nf], t[nf + z:])."""
    y = np.asarray(D, np.float64)
    t = np.roll(np.concatenate([y, -y[::-1]]), -(nf // 2))
    t[3 * nf // 2:] *= -1.0
    t = t / math.sqrt(2.0 * nf) * w[::-1].astype(np.float64)
    return t[z:z + nf], t[nf + z:]


@pytest.mark.parametrize("fs,ms", GEOMETRIES)
def test_engine_unfold_window_and_overlap_add(fs, ms):
    """The engine's unfold with the folded window win = gain * w (one f32 product per sample, where the reference
    rounds t * gain and then * w): every sample equals D * win rounded once, lies within 3 * 2^-24 relative of the float64
    restatement, and the engine-mode DecMdct adds it to the previous frame's tail as overlap_add (:138-151) does."""
    cfg = O.config(fs, ms)
    nf, z = cfg["nf"], cfg["z"]
    sf, fd = _sf_fd(fs, ms)
    win, w, _, _ = _tables(fs, ms)
    gain = np.float32(1.0) / np.sqrt(np.float32(2 * nf))
    assert np.array_equal(win, gain * w[::-1])
    rng = np.random.default_rng(nf + z)
    lib = O.lib()
    for _ in range(8):
        D = rng.standard_normal(nf).astype(np.float32) * np.float32(1000.0)
        head, tail = np.zeros(nf, np.float32), np.zeros(nf - z, np.float32)
        lib.lc3o_engine_unfold(sf, fd, O.p(D), O.p(head), O.p(tail))
        h64, t64 = _unfold64(D, nf, z, w)
        # f32 restatement: the unfolded D (exact, sign flips only) times win, rounded once
        t32 = np.roll(np.concatenate([D, -D[::-1]]), -(nf // 2))
        t32[3 * nf // 2:] *= -1
        assert np.array_equal(head.view(np.uint32), (t32[z:z + nf] * win[z:z + nf]).view(np.uint32))
        assert np.array_equal(tail.view(np.uint32), (t32[nf + z:] * win[nf + z:]).view(np.uint32))
        for got, ref in ((head, h64), (tail, t64)):
            assert (np.abs(got - ref) <= 3 * 2.0 ** -24 * np.abs(ref) + 1e-30).all()
    # overlap-add through the engine-mode DecMdct, two frames: out = mem + head for n < nf - z, head above
    mdct = lib.lc3o_decmdct_new_ex(sf, fd, 1)
    ne = cfg["ne"]
    mem = np.zeros(nf - z, np.float64)
    for f in range(3):
        spec = (rng.standard_normal(ne) * 300.0).astype(np.float32)
        out = np.zeros(nf, np.float32)
        lib.lc3o_decmdct_run(mdct, O.p(spec), O.p(out))
        padded = np.zeros(nf, np.float32)
        padded[:ne] = spec
        h64, t64 = _unfold64(_engine(padded, fs, ms), nf, z, w)
        exp = h64.copy()
        exp[:nf - z] += mem
        err = np.abs(out - exp)
        assert (err <= 4 * 2.0 ** -24 * (np.abs(h64) + np.abs(np.pad(mem, (0, z)))) + 1e-30).all(), (fs, ms, f)
        mem = t64
    lib.lc3o_decmdct_free(mdct)


def _narrowing_is_robust(v, ulps=4):
    """f32(v) is the same for every f64 within +-ulps ulp of v."""
    f = np.float32(v)
    for direction in (math.inf, -math.inf):
        u = v
        for _ in range(ulps):
            u = math.nextafter(u, direction)
            if np.float32(u) != f:
                return False
    return True


@pytest.mark.parametrize("nf", sorted(NF_CONFIG))
def test_twiddle_tables_narrow_the_same_everywhere(nf):
    """init_tables_kernel computes the twiddles with the device's f64 cos / sin (within 2 ulp) and narrows them to f32.
    Every entry's f64 value can move by +-4 ulp without changing its f32 narrowing, so the device's tables equal the
    host's (and the oracle's engine mode) whatever the libm: no entry is at risk at any size."""
    fs, ms = NF_CONFIG[nf]
    _, _, dtw, ftw = _tables(fs, ms)
    N = nf // 2
    at_risk = []
    for i in range(N):
        t = -math.pi * (8 * i + 1) / (8.0 * N * 2.0)
        ph = -2.0 * math.pi * i / N
        for name, table, ang in (("dtw", dtw, t), ("ftw", ftw, ph)):
            for part, fn in ((0, math.cos), (1, math.sin)):
                v = fn(ang)
                assert table[i, part] == np.float32(v), (name, i, part)
                if not _narrowing_is_robust(v):
                    at_risk.append((name, i, part))
    assert at_risk == []


@pytest.mark.parametrize("fs,ms", [(48000, 10), (16000, 7.5), (24000, 10), (32000, 7.5), (8000, 10)])
def test_engine_mode_changes_only_the_transform(fs, ms):
    """Corpus streams with lost frames and garbage frames mixed in: the oracle's engine mode and reference mode give
    identical traces, integer spectra and shaped spectra, and PCM within +-1 LSB.  Prints the fraction of samples that
    differ."""
    nb = MIXED_NBYTES[(fs, ms)]
    _, frames = corpus(fs, ms, nb, 48, 40)
    frames = frames.copy()
    rng = np.random.default_rng(23)
    lens = np.full(frames.shape[:2], nb, np.int32)
    lens[rng.random(lens.shape) < 0.08] = 0
    lens[3, 5:25] = 0                                                   # a 20-frame loss: the fade reaches 0.85
    bad = rng.random(lens.shape) < 0.05
    frames[bad] = rng.integers(0, 256, (int(bad.sum()), nb), dtype=np.uint8)
    r_pcm, r_tr, r_x, r_sp = O.decode_streams(frames, fs, ms, lens, trace=True)
    e_pcm, e_tr, e_x, e_sp = O.decode_streams(frames, fs, ms, lens, trace=True, transform="engine")
    assert np.array_equal(r_tr, e_tr) and np.array_equal(r_x, e_x)
    assert np.array_equal(r_sp.view(np.uint32), e_sp.view(np.uint32))
    assert (r_tr[..., 0] == 0).mean() > 0.05
    d = np.abs(r_pcm.astype(np.int32) - e_pcm.astype(np.int32))
    print(f"{fs} Hz {ms} ms: {100.0 * (d != 0).mean():.3f} % of samples differ by 1 LSB")
    assert d.max() <= 1
    assert (d != 0).any()                                               # the two transforms are not the same function
