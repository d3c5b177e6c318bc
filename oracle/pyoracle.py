"""ctypes binding of the CPU oracle (oracle/_build/liblc3oracle.so).

TEST INFRASTRUCTURE: imported only by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package (lc3_codec_b200) never imports it.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

_DIR = Path(__file__).resolve().parent
_SO = _DIR / "_build" / "liblc3oracle.so"

SF = {8000: 0, 16000: 1, 24000: 2, 32000: 3, 44100: 4, 48000: 5}
FD = {7.5: 0, 10: 1, 10.0: 1}
TRACE_WORDS = 48
# indices into a trace record (mirrors lc3o_capi.cpp / include/lc3b.h)
TR = dict(OK=0, BW=1, LASTNZ=2, LSB_MODE=3, GG_IND=4, NUM_TNS=5, RC_ORDER_IN0=6, RC_ORDER_IN1=7, IND_LF=8, IND_HF=9,
          LS_INDA=10, LS_INDB=11, IDX_A=12, IDX_B=13, SUBMODE_LSB=14, SUBMODE_MSB=15, G_IND=16, PITCH_PRESENT=17,
          LTPF_ACTIVE=18, PITCH_INDEX=19, NOISE_FACTOR=20, RC_ORDER0=21, RC_ORDER1=22, RC_I0=23, NRES=39, SEED=40,
          IS_ZERO=41)


def build(force: bool = False) -> Path:
    srcs = list(_DIR.glob("*.cpp")) + [_DIR / "lc3o.h", _DIR.parent / "lc3_codec_b200" / "csrc" / "lc3_tables.h"]
    stale = (not _SO.exists()) or any(s.stat().st_mtime > _SO.stat().st_mtime for s in srcs if s.exists())
    if force or stale:
        subprocess.run(["make", "-C", str(_DIR)], check=True, capture_output=True)
    return _SO


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(str(_SO))
        for name in ("lc3o_powf",):
            getattr(_lib, name).restype = C.c_float
            getattr(_lib, name).argtypes = [C.c_float, C.c_float]
        for name in ("lc3o_log2f", "lc3o_log10f", "lc3o_exp2f", "lc3o_asinf", "lc3o_sinf", "lc3o_exp2_raw"):
            getattr(_lib, name).restype = C.c_float
            getattr(_lib, name).argtypes = [C.c_float]
        _lib.lc3o_powi.restype = C.c_float
        _lib.lc3o_powi.argtypes = [C.c_float, C.c_int]
        for name in ("lc3o_plc_new", "lc3o_decmdct_new", "lc3o_decltpf_new", "lc3o_decoder_new", "lc3o_encmdct_new",
                     "lc3o_attack_new", "lc3o_encltpf_new", "lc3o_quant_new", "lc3o_encoder_new", "lc3o_decmdct_new_ex"):
            getattr(_lib, name).restype = C.c_void_p
    return _lib


def p(a: np.ndarray):
    """numpy array -> void* (array must stay alive for the call)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(C.c_void_p)


def config(fs: int, ms: float) -> dict:
    out = np.zeros(7, np.int32)
    lib().lc3o_config(SF[fs], FD[ms], p(out))
    return dict(fs_ind=int(out[0]), fs=int(out[1]), ne=int(out[2]), nb=int(out[3]), nf=int(out[4]), z=int(out[5]))


def ncores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def encode_streams(pcm: np.ndarray, fs: int, ms: float, nbytes: int, nthreads: int | None = None) -> np.ndarray:
    """pcm [n_streams, n_frames, nf] i16 -> bytes [n_streams, n_frames, nbytes] u8 (oracle encoder, one channel per stream)."""
    pcm = np.ascontiguousarray(pcm, np.int16)
    s, f, nf = pcm.shape
    assert nf == config(fs, ms)["nf"]
    out = np.zeros((s, f, nbytes), np.uint8)
    lib().lc3o_encode_streams(C.c_int(nthreads or ncores()), s, f, None, SF[fs], FD[ms], p(pcm), nf, p(out), nbytes)
    return out


TRANSFORMS = {"reference": 0, "engine": 1}


def decode_streams(frames: np.ndarray, fs: int, ms: float, nbytes_per_frame: np.ndarray | None = None,
                   nthreads: int | None = None, trace: bool = False, transform: str = "reference"):
    """bytes [n_streams, n_frames, nbytes] u8 -> pcm [n_streams, n_frames, nf] i16 (+ trace, x, spectrum) via the oracle decoder.

    transform = "reference": the reference's inverse MDCT (kissfft DCT-IV, then gain, then window).  "engine": the CUDA
    engine's (its Stockham DCT-IV, unfold and folded window, oracle/lc3o_engine_imdct.cpp); everything else is the
    oracle's own code, so the engine's PCM must equal this bit for bit."""
    frames = np.ascontiguousarray(frames, np.uint8)
    s, f, nb = frames.shape
    cfg = config(fs, ms)
    pcm = np.zeros((s, f, cfg["nf"]), np.int16)
    tr = np.zeros((s, f, TRACE_WORDS), np.int32) if trace else None
    xo = np.zeros((s, f, cfg["ne"]), np.int32) if trace else None
    sp = np.zeros((s, f, cfg["ne"]), np.float32) if trace else None
    npf = None if nbytes_per_frame is None else np.ascontiguousarray(nbytes_per_frame, np.int32)
    if transform == "reference":
        lib().lc3o_decode_streams(C.c_int(nthreads or ncores()), s, f, SF[fs], FD[ms], p(frames), nb, p(npf), p(pcm), p(tr),
                                  p(xo), p(sp))
    else:
        lib().lc3o_decode_streams_ex(C.c_int(nthreads or ncores()), s, f, SF[fs], FD[ms], p(frames), nb, p(npf), p(pcm),
                                     p(tr), p(xo), p(sp), TRANSFORMS[transform])
    return (pcm, tr, xo, sp) if trace else pcm
