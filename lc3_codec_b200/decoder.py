"""Batched mirror of the reference's `Lc3Decoder` (src/decoder/lc3_decoder.rs:51, :180-245).

Reference                                   here
------------------------------------------  -----------------------------------------------------------------
Lc3Decoder::calc_working_buffer_lengths     Lc3BatchDecoder.calc_working_buffer_lengths  (bytes of device workspace)
Lc3Decoder::new(num_channels, ..bufs)       Lc3BatchDecoder(num_streams, .., workspace)  (caller-owned torch buffer)
decode_frame(bits, channel, buf_in, out)    decode_frames(bits, frames, pcm_out, ..)     one frame for EVERY stream
  the same for some channels only           decode_frames_subset(bits, stream_ids, ..)   one frame for each listed stream
  many frames of some channels              decode_stream_frames_subset(bits, ids, counts, ..) counts[i] frames of ids[i]
fresh channel state (Lc3Decoder::new)       reset_streams(stream_ids)                    for the listed streams only
Err(Only16BitsPerAudioSampleSupported)      raises Lc3DecoderError("Only16BitsPerAudioSampleSupported")
panic on bad channel index / slice length   raises Lc3bError(LC3B_ERR_INVALID_ARG)
bitstream errors -> concealment, Ok(())     same; optional `status_out` exposes which streams were concealed
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import native
from .native import FrameDuration, Lc3bError, SamplingFrequency

TRACE_WORDS = 48


class Lc3DecoderError(Exception):
    """Mirror of `Lc3DecoderError` (lc3_decoder.rs:37); only one variant is ever produced (:80)."""


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class Lc3BatchDecoder:
    @staticmethod
    def calc_working_buffer_lengths(num_streams: int, frame_duration: FrameDuration,
                                    sampling_frequency: SamplingFrequency, max_nbytes: int = 400) -> int:
        n = C.c_size_t(0)
        rc = native.lib().lc3b_decoder_workspace_bytes(num_streams, int(frame_duration), int(sampling_frequency),
                                                       max_nbytes, C.byref(n))
        if rc:
            raise Lc3bError(rc, "lc3b_decoder_workspace_bytes")
        return n.value

    def __init__(self, num_streams: int, frame_duration: FrameDuration, sampling_frequency: SamplingFrequency,
                 workspace: torch.Tensor, max_nbytes: int = 400):
        if not workspace.is_cuda or workspace.dtype != torch.uint8:
            raise Lc3bError(2, "workspace must be a CUDA uint8 tensor")
        self.num_streams = num_streams
        self.config = native.config(sampling_frequency, frame_duration)
        self.nf, self.ne = self.config.nf, self.config.ne
        self.max_nbytes = max_nbytes
        self.workspace = workspace                       # borrowed for the decoder's lifetime, like the reference's 'a
        self.device = workspace.device
        self._h = C.c_void_p()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        rc = native.lib().lc3b_decoder_init(C.byref(self._h), num_streams, int(frame_duration), int(sampling_frequency),
                                            max_nbytes, self.device.index or 0, _ptr(workspace),
                                            workspace.numel(), C.c_void_p(stream))
        if rc:
            raise Lc3bError(rc, "lc3b_decoder_init")
        self._trace = None

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            native.lib().lc3b_decoder_destroy(h)

    # ------------------------------------------------------------------ decode_frame, batched
    def decode_frames(self, num_bits_per_audio_sample: int, frames: torch.Tensor, pcm_out: torch.Tensor,
                      frame_nbytes: torch.Tensor | None = None, nbytes: int | None = None,
                      status_out: torch.Tensor | None = None) -> None:
        """frames: CUDA uint8 [num_streams, stride]; pcm_out: CUDA int16 [num_streams, >= nf]."""
        self._call(native.lib().lc3b_decode_frames, True, num_bits_per_audio_sample, frames, pcm_out, frame_nbytes,
                   nbytes, status_out)

    def decode_frames_host(self, num_bits_per_audio_sample: int, frames: torch.Tensor, pcm_out: torch.Tensor,
                           frame_nbytes: torch.Tensor | None = None, nbytes: int | None = None,
                           status_out: torch.Tensor | None = None) -> None:
        """Same with HOST tensors (pin them for asynchronous copies); copies ride the current CUDA stream."""
        self._call(native.lib().lc3b_decode_frames_host, False, num_bits_per_audio_sample, frames, pcm_out,
                   frame_nbytes, nbytes, status_out)

    def decode_frames_subset(self, num_bits_per_audio_sample: int, stream_ids, frames: torch.Tensor, pcm_out: torch.Tensor,
                             frame_nbytes: torch.Tensor | None = None, nbytes: int | None = None,
                             status_out: torch.Tensor | None = None) -> None:
        """decode_frame for the listed streams only; every other stream is untouched (include/lc3b.h).
        stream_ids: host ids (sequence, numpy array or CPU int32 tensor), any order, each at most once; row i of frames,
        pcm_out, frame_nbytes and status_out (CUDA tensors with n_rows = len(stream_ids) rows) belongs to stream_ids[i]."""
        self._call(native.lib().lc3b_decode_frames_subset, True, num_bits_per_audio_sample, frames, pcm_out, frame_nbytes,
                   nbytes, status_out, native.host_ids(stream_ids))

    def reset_streams(self, stream_ids) -> None:
        """Give the listed streams the state a freshly initialised decoder has; no other stream is touched."""
        ids = native.host_ids(stream_ids)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            rc = native.lib().lc3b_decoder_reset_streams(self._h, C.c_void_p(ids.ctypes.data), ids.size, C.c_void_p(stream))
        if rc:
            raise Lc3bError(rc, "lc3b_decoder_reset_streams")

    def _call(self, fn, want_cuda, bits, frames, pcm_out, frame_nbytes, nbytes, status_out, ids=None):
        if bits != 16:
            raise Lc3DecoderError("Only16BitsPerAudioSampleSupported")
        rows = self.num_streams if ids is None else ids.size
        for t, dt, what in ((frames, torch.uint8, "frames"), (pcm_out, torch.int16, "pcm_out")):
            if t.is_cuda != want_cuda or t.dtype != dt or t.dim() != 2 or t.shape[0] != rows or t.stride(1) != 1:
                raise Lc3bError(2, f"{what}: wrong device/dtype/shape")
        if pcm_out.shape[1] < self.nf:
            raise Lc3bError(2, f"pcm_out: {pcm_out.shape[1]} samples per stream, need nf = {self.nf}")
        for t, what in ((frame_nbytes, "frame_nbytes"), (status_out, "status_out")):
            if t is not None and (t.is_cuda != want_cuda or t.dtype != torch.int32 or t.numel() != rows
                                  or not t.is_contiguous()):
                raise Lc3bError(2, f"{what}: wrong device/dtype/shape")
        nb = frames.shape[1] if nbytes is None else nbytes
        head = () if ids is None else (C.c_void_p(ids.ctypes.data), ids.size)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            rc = fn(self._h, bits, *head, _ptr(frames), _ptr(frame_nbytes), nb, frames.stride(0), _ptr(pcm_out),
                    pcm_out.stride(0), _ptr(status_out), C.c_void_p(stream))
        if rc == 1:
            raise Lc3DecoderError("Only16BitsPerAudioSampleSupported")
        if rc:
            raise Lc3bError(rc, fn.__name__)

    # ------------------------------------------------------------------ time-parallel decode (SURVEY.md 8f-1)
    def multi_scratch_bytes(self, n_frames: int) -> int:
        n = C.c_size_t(0)
        rc = native.lib().lc3b_decoder_multi_scratch_bytes(self._h, n_frames, C.byref(n))
        if rc:
            raise Lc3bError(rc, "lc3b_decoder_multi_scratch_bytes")
        return int(n.value)

    def decode_stream_frames(self, num_bits_per_audio_sample: int, frames: torch.Tensor, pcm_out: torch.Tensor,
                             scratch: torch.Tensor, frame_nbytes: torch.Tensor | None = None,
                             status_out: torch.Tensor | None = None) -> None:
        """Many consecutive frames of every stream in one call (the file workflow of examples/decode.rs).
        frames: CUDA uint8 [num_streams, n_frames, nbytes] contiguous; pcm_out: CUDA int16 [num_streams, n_frames * nf];
        scratch: CUDA uint8, >= multi_scratch_bytes(n_frames); frame_nbytes / status_out: CUDA int32 [num_streams, n_frames]."""
        if num_bits_per_audio_sample != 16:
            raise Lc3DecoderError("Only16BitsPerAudioSampleSupported")
        if not (frames.is_cuda and frames.dtype == torch.uint8 and frames.dim() == 3 and frames.shape[0] == self.num_streams
                and frames.is_contiguous()):
            raise Lc3bError(2, "frames: want contiguous CUDA uint8 [num_streams, n_frames, nbytes]")
        F, nb = frames.shape[1], frames.shape[2]
        if not (pcm_out.is_cuda and pcm_out.dtype == torch.int16 and pcm_out.is_contiguous()
                and pcm_out.numel() == self.num_streams * F * self.nf):
            raise Lc3bError(2, "pcm_out: want contiguous CUDA int16 [num_streams, n_frames * nf]")
        for t, what in ((frame_nbytes, "frame_nbytes"), (status_out, "status_out")):
            if t is not None and not (t.is_cuda and t.dtype == torch.int32 and t.numel() == self.num_streams * F and t.is_contiguous()):
                raise Lc3bError(2, f"{what}: wrong device/dtype/shape")
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            rc = native.lib().lc3b_decode_stream_frames(self._h, 16, _ptr(frames), _ptr(frame_nbytes), nb, nb, F, _ptr(pcm_out),
                                                        _ptr(status_out), _ptr(scratch), scratch.numel(), C.c_void_p(stream))
        if rc:
            raise Lc3bError(rc, "lc3b_decode_stream_frames")

    def multi_subset_scratch_bytes(self, n_rows: int, total_frames: int) -> int:
        """Bytes of caller-owned device scratch decode_stream_frames_subset needs for n_rows rows and total_frames frames."""
        n = C.c_size_t(0)
        rc = native.lib().lc3b_decoder_multi_subset_scratch_bytes(self._h, int(n_rows), int(total_frames), C.byref(n))
        if rc:
            raise Lc3bError(rc, "lc3b_decoder_multi_subset_scratch_bytes")
        return int(n.value)

    def decode_stream_frames_subset(self, num_bits_per_audio_sample: int, stream_ids, frame_counts, frames: torch.Tensor,
                                    pcm_out: torch.Tensor, scratch: torch.Tensor, frame_nbytes: torch.Tensor | None = None,
                                    status_out: torch.Tensor | None = None) -> None:
        """frame_counts[i] consecutive frames of stream stream_ids[i] in one call, equal to that many decode_frames calls on
        it; streams not listed are untouched (include/lc3b.h).  stream_ids, frame_counts: host sequences, numpy arrays or
        CPU int32 tensors of one length.  The rows' frames are packed row after row in the caller's order (V = sum of the
        counts): frames: contiguous CUDA uint8 [V, nbytes]; pcm_out: contiguous CUDA int16 with V * nf samples;
        scratch: CUDA uint8, >= multi_subset_scratch_bytes(len(stream_ids), V); frame_nbytes / status_out: CUDA int32 [V]."""
        if num_bits_per_audio_sample != 16:
            raise Lc3DecoderError("Only16BitsPerAudioSampleSupported")
        ids = native.host_ids(stream_ids)
        counts = native.host_counts(frame_counts, ids.size)
        V = int(counts.astype(np.int64).sum()) if counts.size else 0
        if not (frames.is_cuda and frames.dtype == torch.uint8 and frames.dim() == 2 and frames.shape[0] == V
                and frames.is_contiguous()):
            raise Lc3bError(2, f"frames: want contiguous CUDA uint8 [{V}, nbytes]")
        nb = frames.shape[1]
        if not (pcm_out.is_cuda and pcm_out.dtype == torch.int16 and pcm_out.is_contiguous() and pcm_out.numel() == V * self.nf):
            raise Lc3bError(2, f"pcm_out: want contiguous CUDA int16 with {V} * nf samples")
        for t, what in ((frame_nbytes, "frame_nbytes"), (status_out, "status_out")):
            if t is not None and not (t.is_cuda and t.dtype == torch.int32 and t.numel() == V and t.is_contiguous()):
                raise Lc3bError(2, f"{what}: wrong device/dtype/shape")
        if not (scratch.is_cuda and scratch.dtype == torch.uint8):
            raise Lc3bError(2, "scratch must be a CUDA uint8 tensor")
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            rc = native.lib().lc3b_decode_stream_frames_subset(
                self._h, 16, C.c_void_p(ids.ctypes.data), C.c_void_p(counts.ctypes.data), ids.size, _ptr(frames),
                _ptr(frame_nbytes), nb, nb, _ptr(pcm_out), _ptr(status_out), _ptr(scratch), scratch.numel(), C.c_void_p(stream))
        if rc:
            raise Lc3bError(rc, "lc3b_decode_stream_frames_subset")

    # ------------------------------------------------------------------ inspection (parity gate i)
    def enable_trace(self):
        """Allocates and registers device buffers for the per-frame inspection record and integer spectrum."""
        tr = torch.zeros((self.num_streams, TRACE_WORDS), dtype=torch.int32, device=self.device)
        x = torch.zeros((self.num_streams, self.ne), dtype=torch.int32, device=self.device)
        rc = native.lib().lc3b_decoder_set_trace(self._h, _ptr(tr), _ptr(x))
        if rc:
            raise Lc3bError(rc, "lc3b_decoder_set_trace")
        self._trace = (tr, x)
        return tr, x

    def set_host_pipelining(self, on: bool) -> None:
        """Overlap the PCM device->host copy of call i with the kernels of call i+1 (see include/lc3b.h)."""
        rc = native.lib().lc3b_decoder_set_host_pipelining(self._h, int(bool(on)))
        if rc:
            raise Lc3bError(rc, "lc3b_decoder_set_host_pipelining")

    def host_fence(self) -> None:
        """Make the current CUDA stream wait for every outstanding pipelined PCM copy."""
        stream = torch.cuda.current_stream(self.device).cuda_stream
        rc = native.lib().lc3b_decoder_host_fence(self._h, C.c_void_p(stream))
        if rc:
            raise Lc3bError(rc, "lc3b_decoder_host_fence")

    def set_graph_mode(self, on: bool) -> None:
        """Issue every call as ONE cached CUDA graph launch (True) or one launch per kernel (False); include/lc3b.h."""
        rc = native.lib().lc3b_decoder_set_graph_mode(self._h, int(bool(on)))
        if rc:
            raise Lc3bError(rc, "lc3b_decoder_set_graph_mode")

    def set_split(self, k: int) -> None:
        """Cut every call into k independent sub-batches whose kernels overlap (0 = by batch size, 1 = never, 2, 4); include/lc3b.h."""
        rc = native.lib().lc3b_decoder_set_split(self._h, int(k))
        if rc:
            raise Lc3bError(rc, "lc3b_decoder_set_split")

    def set_min_nbytes(self, min_nbytes: int) -> None:
        """Promise that every submitted frame is at least min_nbytes long (or lost).  When that rules the long-term post filter
        out for good (e.g. >= 110 bytes at 48 kHz / 10 ms) the decoder stops keeping the filter's output history; include/lc3b.h."""
        rc = native.lib().lc3b_decoder_set_min_nbytes(self._h, int(min_nbytes))
        if rc:
            raise Lc3bError(rc, "lc3b_decoder_set_min_nbytes")

    def set_synth_mode(self, mode: int) -> None:
        """0 = synthesis kernel chosen by launch size (default), 1 = one frame per warp always (identical results)."""
        rc = native.lib().lc3b_decoder_set_synth_mode(self._h, mode)
        if rc:
            raise Lc3bError(rc, "lc3b_decoder_set_synth_mode")

    def set_dequant_mode(self, mode: int) -> None:
        """0 = dequantisation kernel chosen by batch size, 1 = warp per frame, 2 = thread per frame (identical results)."""
        rc = native.lib().lc3b_decoder_set_dequant_mode(self._h, mode)
        if rc:
            raise Lc3bError(rc, "lc3b_decoder_set_dequant_mode")

    def graph_stats(self) -> dict:
        a, b, c = C.c_uint64(0), C.c_uint64(0), C.c_uint64(0)
        rc = native.lib().lc3b_decoder_graph_stats(self._h, C.byref(a), C.byref(b), C.byref(c))
        if rc:
            raise Lc3bError(rc, "lc3b_decoder_graph_stats")
        return {"hits": a.value, "updates": b.value, "builds": c.value}

    def set_stage_mask(self, mask: int) -> None:
        """Profiling hook (lc3b_decoder_set_stage_mask): bit 0 = entropy kernel, bit 1 = dequantisation kernel, bit 2 =
        synthesis + post-filter kernels; default 7 (all).  Results are only meaningful with mask 7."""
        rc = native.lib().lc3b_decoder_set_stage_mask(self._h, mask)
        if rc:
            raise Lc3bError(rc, "lc3b_decoder_set_stage_mask")

    def spectrum(self) -> torch.Tensor:
        out = torch.empty((self.num_streams, self.ne), dtype=torch.float32, device=self.device)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        rc = native.lib().lc3b_decoder_get_spectrum(self._h, _ptr(out), C.c_void_p(stream))
        if rc:
            raise Lc3bError(rc, "lc3b_decoder_get_spectrum")
        return out
