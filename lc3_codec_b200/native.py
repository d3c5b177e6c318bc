"""ctypes binding of liblc3b.so (include/lc3b.h).  Fails loudly when the CUDA library is missing."""
from __future__ import annotations

import ctypes as C
import enum
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_SO = _HERE / "liblc3b.so"


class SamplingFrequency(enum.IntEnum):      # src/common/config.rs:2
    Hz8000 = 0
    Hz16000 = 1
    Hz24000 = 2
    Hz32000 = 3
    Hz44100 = 4
    Hz48000 = 5

    @staticmethod
    def from_hz(hz: int) -> "SamplingFrequency":
        return {8000: SamplingFrequency.Hz8000, 16000: SamplingFrequency.Hz16000, 24000: SamplingFrequency.Hz24000,
                32000: SamplingFrequency.Hz32000, 44100: SamplingFrequency.Hz44100, 48000: SamplingFrequency.Hz48000}[hz]


class FrameDuration(enum.IntEnum):          # src/common/config.rs:12
    SevenPointFiveMs = 0
    TenMs = 1

    @staticmethod
    def from_ms(ms: float) -> "FrameDuration":
        if float(ms) == 10.0:
            return FrameDuration.TenMs
        if float(ms) == 7.5:
            return FrameDuration.SevenPointFiveMs
        raise ValueError(f"LC3 frame durations are 7.5 and 10 ms, not {ms}")


class Lc3bError(RuntimeError):
    """A non-zero status from the C ABI (LC3B_ERR_*)."""

    def __init__(self, code: int, what: str):
        names = {1: "LC3B_ERR_BITS_PER_SAMPLE", 2: "LC3B_ERR_INVALID_ARG", 3: "LC3B_ERR_CUDA", 4: "LC3B_ERR_WORKSPACE"}
        extra = f" (cudaError {lib().lc3b_last_cuda_error()})" if code == 3 else ""
        super().__init__(f"{what}: {names.get(code, code)}{extra}")
        self.code = code


class Config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("fs_ind", "fs", "ne", "nb", "nf", "z", "n_ms")]


EXPORTS = ["lc3b_config_new", "lc3b_last_cuda_error", "lc3b_version", "lc3b_decoder_workspace_bytes",
           "lc3b_decoder_init", "lc3b_decode_frames", "lc3b_decode_frames_host", "lc3b_decoder_set_trace",
           "lc3b_decoder_get_spectrum", "lc3b_decoder_set_stage_mask", "lc3b_decoder_set_host_pipelining",
           "lc3b_decoder_host_fence", "lc3b_decoder_multi_scratch_bytes", "lc3b_decode_stream_frames", "lc3b_decoder_destroy",
           "lc3b_selftest_math_host",
           "lc3b_selftest_math_device", "lc3b_encoder_workspace_bytes", "lc3b_encoder_init", "lc3b_encode_frames",
           "lc3b_encode_frames_host", "lc3b_encoder_multi_scratch_bytes", "lc3b_encode_stream_frames", "lc3b_encoder_set_host_pipelining", "lc3b_encoder_debug_read", "lc3b_encoder_set_stage_mask",
           "lc3b_encoder_destroy", "lc3b_decoder_set_graph_mode", "lc3b_decoder_set_split", "lc3b_decoder_graph_stats", "lc3b_decoder_set_dequant_mode", "lc3b_mixed_decoder_set_dequant_mode", "lc3b_decoder_set_min_nbytes", "lc3b_decoder_set_synth_mode", "lc3b_encoder_set_graph_mode",
           "lc3b_mixed_decoder_layout", "lc3b_mixed_decoder_workspace_bytes", "lc3b_mixed_decoder_init", "lc3b_mixed_decode_frames",
           "lc3b_mixed_decode_frames_host", "lc3b_mixed_decoder_set_host_pipelining", "lc3b_mixed_decoder_host_fence",
           "lc3b_mixed_decoder_set_graph_mode", "lc3b_mixed_decoder_destroy",
           "lc3b_sharded_decoder_create", "lc3b_sharded_decoder_n_shards", "lc3b_sharded_decoder_shard",
           "lc3b_sharded_decode_frames_host", "lc3b_sharded_decoder_wait", "lc3b_sharded_decoder_set_min_nbytes", "lc3b_sharded_decoder_destroy",
           "lc3b_sharded_encoder_create", "lc3b_sharded_encoder_n_shards", "lc3b_sharded_encoder_shard",
           "lc3b_sharded_encode_frames_host", "lc3b_sharded_encoder_wait", "lc3b_sharded_encoder_destroy",
           "lc3b_host_alloc", "lc3b_host_free",
           "lc3b_decode_frames_subset", "lc3b_decoder_reset_streams", "lc3b_encode_frames_subset", "lc3b_encoder_reset_streams",
           "lc3b_decoder_multi_subset_scratch_bytes", "lc3b_decode_stream_frames_subset",
           "lc3b_encoder_multi_subset_scratch_bytes", "lc3b_encode_stream_frames_subset"]


class MixedBucket(C.Structure):             # lc3b_mixed_bucket
    _fields_ = [("sampling_frequency", C.c_int32), ("frame_duration", C.c_int32), ("first_row", C.c_int32),
                ("n_rows", C.c_int32), ("nf", C.c_int32), ("reserved", C.c_int32), ("host_pcm_offset", C.c_uint64)]

_lib = None


def lib_path() -> Path:
    return _SO


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not _SO.exists():
            raise ImportError(f"{_SO} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(nvcc, sm_100a).  lc3_codec_b200 has no CPU fallback.")
        L = C.CDLL(str(_SO))
        vp, i32, sz = C.c_void_p, C.c_int, C.c_size_t
        L.lc3b_version.restype = C.c_char_p
        L.lc3b_config_new.argtypes = [i32, i32, C.POINTER(Config)]
        L.lc3b_decoder_workspace_bytes.argtypes = [i32, i32, i32, i32, C.POINTER(sz)]
        L.lc3b_decoder_init.argtypes = [C.POINTER(vp), i32, i32, i32, i32, i32, vp, sz, vp]
        L.lc3b_decode_frames.argtypes = [vp, i32, vp, vp, i32, sz, vp, sz, vp, vp]
        L.lc3b_decode_frames_host.argtypes = [vp, i32, vp, vp, i32, sz, vp, sz, vp, vp]
        L.lc3b_decoder_set_trace.argtypes = [vp, vp, vp]
        L.lc3b_decoder_get_spectrum.argtypes = [vp, vp, vp]
        L.lc3b_decoder_set_stage_mask.argtypes = [vp, i32]
        L.lc3b_decoder_set_host_pipelining.argtypes = [vp, i32]
        L.lc3b_decoder_host_fence.argtypes = [vp, vp]
        L.lc3b_decoder_multi_scratch_bytes.argtypes = [vp, i32, C.POINTER(C.c_size_t)]
        L.lc3b_decode_stream_frames.argtypes = [vp, i32, vp, vp, i32, sz, i32, vp, vp, vp, sz, vp]
        L.lc3b_decode_frames_subset.argtypes = [vp, i32, vp, i32, vp, vp, i32, sz, vp, sz, vp, vp]
        L.lc3b_decoder_reset_streams.argtypes = [vp, vp, i32, vp]
        L.lc3b_decoder_multi_subset_scratch_bytes.argtypes = [vp, i32, C.c_longlong, C.POINTER(sz)]
        L.lc3b_decode_stream_frames_subset.argtypes = [vp, i32, vp, vp, i32, vp, vp, i32, sz, vp, vp, vp, sz, vp]
        L.lc3b_decoder_destroy.argtypes = [vp]
        L.lc3b_decoder_destroy.restype = None
        L.lc3b_encoder_workspace_bytes.argtypes = [i32, i32, i32, i32, C.POINTER(sz)]
        L.lc3b_encoder_init.argtypes = [C.POINTER(vp), i32, i32, i32, i32, i32, vp, sz, vp]
        L.lc3b_encode_frames.argtypes = [vp, vp, sz, vp, i32, sz, vp]
        L.lc3b_encode_frames_host.argtypes = [vp, vp, sz, vp, i32, sz, vp]
        L.lc3b_encoder_multi_scratch_bytes.argtypes = [vp, i32, C.POINTER(sz)]
        L.lc3b_encode_stream_frames.argtypes = [vp, vp, i32, vp, i32, sz, vp, sz, vp]
        L.lc3b_encode_frames_subset.argtypes = [vp, vp, i32, vp, sz, vp, i32, sz, vp]
        L.lc3b_encoder_reset_streams.argtypes = [vp, vp, i32, vp]
        L.lc3b_encoder_multi_subset_scratch_bytes.argtypes = [vp, i32, C.c_longlong, C.POINTER(sz)]
        L.lc3b_encode_stream_frames_subset.argtypes = [vp, vp, vp, i32, vp, vp, i32, sz, vp, sz, vp]
        L.lc3b_encoder_debug_read.argtypes = [vp, vp, vp, vp, vp, vp]
        L.lc3b_encoder_set_stage_mask.argtypes = [vp, i32]
        L.lc3b_encoder_set_host_pipelining.argtypes = [vp, i32]
        L.lc3b_encoder_destroy.argtypes = [vp]
        L.lc3b_encoder_destroy.restype = None
        u64p, i32p = C.POINTER(C.c_uint64), C.POINTER(C.c_int32)
        L.lc3b_decoder_set_graph_mode.argtypes = [vp, i32]
        L.lc3b_decoder_set_split.argtypes = [vp, i32]
        L.lc3b_decoder_set_dequant_mode.argtypes = [vp, i32]
        L.lc3b_decoder_set_min_nbytes.argtypes = [vp, i32]
        L.lc3b_decoder_set_synth_mode.argtypes = [vp, i32]
        L.lc3b_mixed_decoder_set_dequant_mode.argtypes = [vp, i32]
        L.lc3b_decoder_graph_stats.argtypes = [vp, u64p, u64p, u64p]
        L.lc3b_encoder_set_graph_mode.argtypes = [vp, i32]
        L.lc3b_mixed_decoder_layout.argtypes = [i32, vp, vp, vp, C.POINTER(MixedBucket), i32p, u64p]
        L.lc3b_mixed_decoder_workspace_bytes.argtypes = [i32, vp, vp, i32, C.POINTER(sz)]
        L.lc3b_mixed_decoder_init.argtypes = [C.POINTER(vp), i32, vp, vp, i32, i32, vp, sz, vp]
        L.lc3b_mixed_decode_frames.argtypes = [vp, i32, vp, vp, i32, sz, vp, sz, vp, vp]
        L.lc3b_mixed_decode_frames_host.argtypes = [vp, i32, vp, vp, i32, sz, vp, vp, vp]
        L.lc3b_mixed_decoder_set_host_pipelining.argtypes = [vp, i32]
        L.lc3b_mixed_decoder_host_fence.argtypes = [vp, vp]
        L.lc3b_mixed_decoder_set_graph_mode.argtypes = [vp, i32]
        L.lc3b_mixed_decoder_destroy.argtypes = [vp]
        L.lc3b_mixed_decoder_destroy.restype = None
        for kind in ("decoder", "encoder"):
            getattr(L, f"lc3b_sharded_{kind}_create").argtypes = [C.POINTER(vp), i32, i32, i32, i32, i32p, i32]
            getattr(L, f"lc3b_sharded_{kind}_n_shards").argtypes = [vp]
            getattr(L, f"lc3b_sharded_{kind}_shard").argtypes = [vp, i32, i32p, i32p, i32p]
            getattr(L, f"lc3b_sharded_{kind}_wait").argtypes = [vp]
            getattr(L, f"lc3b_sharded_{kind}_destroy").argtypes = [vp]
            getattr(L, f"lc3b_sharded_{kind}_destroy").restype = None
        L.lc3b_sharded_decoder_set_min_nbytes.argtypes = [vp, i32]
        L.lc3b_sharded_decode_frames_host.argtypes = [vp, i32, vp, vp, i32, sz, vp, sz, vp]
        L.lc3b_sharded_encode_frames_host.argtypes = [vp, vp, sz, vp, i32, sz]
        L.lc3b_host_alloc.argtypes = [C.POINTER(vp), sz]
        L.lc3b_host_free.argtypes = [vp]
        L.lc3b_host_free.restype = None
        L.lc3b_selftest_math_host.argtypes = [i32, vp, vp, vp, i32]
        L.lc3b_selftest_math_device.argtypes = [i32, vp, vp, vp, i32, vp]
        _lib = L
    return _lib


def host_ids(stream_ids) -> np.ndarray:
    """A subset call's id list (a sequence, a numpy array or a CPU int32 tensor) as a contiguous host int32 array.
    Range and uniqueness are checked by the library."""
    if hasattr(stream_ids, "is_cuda"):                 # a torch tensor
        if stream_ids.is_cuda or str(stream_ids.dtype) != "torch.int32" or stream_ids.dim() != 1:
            raise Lc3bError(2, "stream_ids: want a 1-D CPU int32 tensor")
        stream_ids = stream_ids.contiguous().numpy()
    a = np.asarray(stream_ids)
    if a.ndim != 1 or (a.size and a.dtype.kind not in "iu"):
        raise Lc3bError(2, "stream_ids: want a 1-D sequence of integers")
    if a.size and (int(a.min()) < -2**31 or int(a.max()) >= 2**31):
        raise Lc3bError(2, "stream_ids: ids beyond int32")
    return np.ascontiguousarray(a, dtype=np.int32)


def host_counts(frame_counts, n_rows: int) -> np.ndarray:
    """A ragged call's frame counts (a sequence, a numpy array or a CPU int32 tensor), one per row of its id list, as a
    contiguous host int32 array.  Signs and the total are checked by the library."""
    if hasattr(frame_counts, "is_cuda"):               # a torch tensor
        if frame_counts.is_cuda or str(frame_counts.dtype) != "torch.int32" or frame_counts.dim() != 1:
            raise Lc3bError(2, "frame_counts: want a 1-D CPU int32 tensor")
        frame_counts = frame_counts.contiguous().numpy()
    a = np.asarray(frame_counts)
    if a.ndim != 1 or (a.size and a.dtype.kind not in "iu"):
        raise Lc3bError(2, "frame_counts: want a 1-D sequence of integers")
    if a.size != n_rows:
        raise Lc3bError(2, f"frame_counts: {a.size} counts for {n_rows} stream ids")
    if a.size and (int(a.min()) < -2**31 or int(a.max()) >= 2**31):
        raise Lc3bError(2, "frame_counts: counts beyond int32")
    return np.ascontiguousarray(a, dtype=np.int32)


def config(sampling_frequency: int, frame_duration: int) -> Config:
    c = Config()
    rc = lib().lc3b_config_new(int(sampling_frequency), int(frame_duration), C.byref(c))
    if rc:
        raise Lc3bError(rc, "lc3b_config_new")
    return c
