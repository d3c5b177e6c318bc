"""Batched mirror of the reference's `Lc3Encoder` (src/encoder/lc3_encoder.rs:33, :116-210).

Reference                                   here
------------------------------------------  -----------------------------------------------------------------
Lc3Encoder::calc_working_buffer_lengths     Lc3BatchEncoder.calc_working_buffer_lengths  (bytes of device workspace)
Lc3Encoder::new(num_channels, ..bufs)       Lc3BatchEncoder(num_streams, .., workspace)
encode_frame(channel, samples_in, buf_out)  encode_frames(pcm_in, frames_out)            one frame for EVERY stream
  the same for some channels only           encode_frames_subset(stream_ids, ..)         one frame for each listed stream
  many frames of some channels              encode_stream_frames_subset(ids, counts, ..) counts[i] frames of ids[i]
fresh channel state (Lc3Encoder::new)       reset_streams(stream_ids)                    for the listed streams only
Result<(), Lc3EncoderError> (empty enum)    returns None; cannot fail for valid shapes
assert_eq!(samples_in.len(), nf) panics     raises Lc3bError(LC3B_ERR_INVALID_ARG)
Lc3Encoder::new panics at 8 kHz             raises Lc3bError(LC3B_ERR_INVALID_ARG)
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import native
from .native import FrameDuration, Lc3bError, SamplingFrequency


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class Lc3BatchEncoder:
    @staticmethod
    def calc_working_buffer_lengths(num_streams: int, frame_duration: FrameDuration,
                                    sampling_frequency: SamplingFrequency, max_nbytes: int = 400) -> int:
        n = C.c_size_t(0)
        rc = native.lib().lc3b_encoder_workspace_bytes(num_streams, int(frame_duration), int(sampling_frequency),
                                                       max_nbytes, C.byref(n))
        if rc:
            raise Lc3bError(rc, "lc3b_encoder_workspace_bytes")
        return n.value

    def __init__(self, num_streams: int, frame_duration: FrameDuration, sampling_frequency: SamplingFrequency,
                 workspace: torch.Tensor, max_nbytes: int = 400):
        if not workspace.is_cuda or workspace.dtype != torch.uint8:
            raise Lc3bError(2, "workspace must be a CUDA uint8 tensor")
        self.num_streams = num_streams
        self.config = native.config(sampling_frequency, frame_duration)
        self.nf, self.ne = self.config.nf, self.config.ne
        self.max_nbytes = max_nbytes
        self.workspace = workspace
        self.device = workspace.device
        self._h = C.c_void_p()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        rc = native.lib().lc3b_encoder_init(C.byref(self._h), num_streams, int(frame_duration), int(sampling_frequency),
                                            max_nbytes, self.device.index or 0, _ptr(workspace), workspace.numel(),
                                            C.c_void_p(stream))
        if rc:
            raise Lc3bError(rc, "lc3b_encoder_init")

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            native.lib().lc3b_encoder_destroy(h)

    def encode_frames(self, pcm_in: torch.Tensor, frames_out: torch.Tensor) -> None:
        """pcm_in: CUDA int16 [num_streams, nf]; frames_out: CUDA uint8 [num_streams, nbytes] (nbytes = buf_out.len())."""
        self._call(native.lib().lc3b_encode_frames, True, pcm_in, frames_out)

    def encode_frames_host(self, pcm_in: torch.Tensor, frames_out: torch.Tensor) -> None:
        self._call(native.lib().lc3b_encode_frames_host, False, pcm_in, frames_out)

    def encode_frames_subset(self, stream_ids, pcm_in: torch.Tensor, frames_out: torch.Tensor) -> None:
        """encode_frame for the listed streams only; every other stream is untouched (include/lc3b.h).
        stream_ids: host ids (sequence, numpy array or CPU int32 tensor), any order, each at most once; row i of pcm_in
        and frames_out (CUDA tensors with n_rows = len(stream_ids) rows) belongs to stream_ids[i]."""
        self._call(native.lib().lc3b_encode_frames_subset, True, pcm_in, frames_out, native.host_ids(stream_ids))

    def reset_streams(self, stream_ids) -> None:
        """Give the listed streams the state a freshly initialised encoder has; no other stream is touched."""
        ids = native.host_ids(stream_ids)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            rc = native.lib().lc3b_encoder_reset_streams(self._h, C.c_void_p(ids.ctypes.data), ids.size, C.c_void_p(stream))
        if rc:
            raise Lc3bError(rc, "lc3b_encoder_reset_streams")

    def _call(self, fn, want_cuda, pcm_in, frames_out, ids=None):
        rows = self.num_streams if ids is None else ids.size
        for t, dt, what in ((pcm_in, torch.int16, "pcm_in"), (frames_out, torch.uint8, "frames_out")):
            if t.is_cuda != want_cuda or t.dtype != dt or t.dim() != 2 or t.shape[0] != rows or t.stride(1) != 1:
                raise Lc3bError(2, f"{what}: wrong device/dtype/shape")
        if pcm_in.shape[1] != self.nf:
            raise Lc3bError(2, f"pcm_in: {pcm_in.shape[1]} samples per stream, need nf = {self.nf}")
        head = () if ids is None else (C.c_void_p(ids.ctypes.data), ids.size)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            rc = fn(self._h, *head, _ptr(pcm_in), pcm_in.stride(0), _ptr(frames_out), frames_out.shape[1], frames_out.stride(0),
                    C.c_void_p(stream))
        if rc:
            raise Lc3bError(rc, fn.__name__)

    # ------------------------------------------------------------------ time-parallel encode
    def multi_scratch_bytes(self, n_frames: int) -> int:
        """Bytes of caller-owned device scratch encode_stream_frames needs for n_frames frames per stream."""
        n = C.c_size_t(0)
        rc = native.lib().lc3b_encoder_multi_scratch_bytes(self._h, n_frames, C.byref(n))
        if rc:
            raise Lc3bError(rc, "lc3b_encoder_multi_scratch_bytes")
        return int(n.value)

    def encode_stream_frames(self, pcm_in: torch.Tensor, frames_out: torch.Tensor, scratch: torch.Tensor) -> None:
        """Many consecutive frames of every stream in one call, equal to n_frames encode_frames calls.
        pcm_in: CUDA int16 [num_streams, n_frames * nf] contiguous; frames_out: CUDA uint8 [num_streams, n_frames, nbytes]
        contiguous; scratch: CUDA uint8, >= multi_scratch_bytes(n_frames)."""
        if not (frames_out.is_cuda and frames_out.dtype == torch.uint8 and frames_out.dim() == 3
                and frames_out.shape[0] == self.num_streams and frames_out.is_contiguous()):
            raise Lc3bError(2, "frames_out: want contiguous CUDA uint8 [num_streams, n_frames, nbytes]")
        F, nb = frames_out.shape[1], frames_out.shape[2]
        if not (pcm_in.is_cuda and pcm_in.dtype == torch.int16 and pcm_in.dim() == 2 and pcm_in.shape[0] == self.num_streams
                and pcm_in.shape[1] == F * self.nf and pcm_in.is_contiguous()):
            raise Lc3bError(2, f"pcm_in: want contiguous CUDA int16 [num_streams, n_frames * nf = {F * self.nf}]")
        if not (scratch.is_cuda and scratch.dtype == torch.uint8):
            raise Lc3bError(2, "scratch must be a CUDA uint8 tensor")
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            rc = native.lib().lc3b_encode_stream_frames(self._h, _ptr(pcm_in), F, _ptr(frames_out), nb, nb, _ptr(scratch),
                                                        scratch.numel(), C.c_void_p(stream))
        if rc:
            raise Lc3bError(rc, "lc3b_encode_stream_frames")

    def multi_subset_scratch_bytes(self, n_rows: int, total_frames: int) -> int:
        """Bytes of caller-owned device scratch encode_stream_frames_subset needs for n_rows rows and total_frames frames."""
        n = C.c_size_t(0)
        rc = native.lib().lc3b_encoder_multi_subset_scratch_bytes(self._h, int(n_rows), int(total_frames), C.byref(n))
        if rc:
            raise Lc3bError(rc, "lc3b_encoder_multi_subset_scratch_bytes")
        return int(n.value)

    def encode_stream_frames_subset(self, stream_ids, frame_counts, pcm_in: torch.Tensor, frames_out: torch.Tensor,
                                    scratch: torch.Tensor) -> None:
        """frame_counts[i] consecutive frames of stream stream_ids[i] in one call, equal to that many encode_frames calls on
        it; streams not listed are untouched (include/lc3b.h).  Frames are packed row after row in the caller's order
        (V = sum of the counts): pcm_in: contiguous CUDA int16 with V * nf samples; frames_out: contiguous CUDA uint8
        [V, nbytes]; scratch: CUDA uint8, >= multi_subset_scratch_bytes(len(stream_ids), V)."""
        ids = native.host_ids(stream_ids)
        counts = native.host_counts(frame_counts, ids.size)
        V = int(counts.astype(np.int64).sum()) if counts.size else 0
        if not (frames_out.is_cuda and frames_out.dtype == torch.uint8 and frames_out.dim() == 2 and frames_out.shape[0] == V
                and frames_out.is_contiguous()):
            raise Lc3bError(2, f"frames_out: want contiguous CUDA uint8 [{V}, nbytes]")
        nb = frames_out.shape[1]
        if not (pcm_in.is_cuda and pcm_in.dtype == torch.int16 and pcm_in.is_contiguous() and pcm_in.numel() == V * self.nf):
            raise Lc3bError(2, f"pcm_in: want contiguous CUDA int16 with {V} * nf samples")
        if not (scratch.is_cuda and scratch.dtype == torch.uint8):
            raise Lc3bError(2, "scratch must be a CUDA uint8 tensor")
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            rc = native.lib().lc3b_encode_stream_frames_subset(
                self._h, C.c_void_p(ids.ctypes.data), C.c_void_p(counts.ctypes.data), ids.size, _ptr(pcm_in), _ptr(frames_out),
                nb, nb, _ptr(scratch), scratch.numel(), C.c_void_p(stream))
        if rc:
            raise Lc3bError(rc, "lc3b_encode_stream_frames_subset")

    def set_host_pipelining(self, on: bool) -> None:
        """Let the PCM upload of encode_frames_host call i+1 overlap the kernels of call i (include/lc3b.h)."""
        rc = native.lib().lc3b_encoder_set_host_pipelining(self._h, 1 if on else 0)
        if rc != 0:
            raise Lc3bError(rc, "lc3b_encoder_set_host_pipelining")

    def set_graph_mode(self, on: bool) -> None:
        """Issue every call as ONE cached CUDA graph launch (True) or one launch per kernel (False); include/lc3b.h."""
        rc = native.lib().lc3b_encoder_set_graph_mode(self._h, int(bool(on)))
        if rc:
            raise Lc3bError(rc, "lc3b_encoder_set_graph_mode")

    def set_stage_mask(self, mask: int) -> None:
        """Profiling hook (lc3b_encoder_set_stage_mask): bit 0 = MDCT kernel, bit 1 = attack / LTPF analysis kernel,
        bit 2 = SNS kernel, bit 3 = TNS kernel, bit 4 = quantise kernel, bit 5 = bitstream stage; default 63 (all)."""
        rc = native.lib().lc3b_encoder_set_stage_mask(self._h, mask)
        if rc:
            raise Lc3bError(rc, "lc3b_encoder_set_stage_mask")

    def debug_read(self):
        """(xf, e_b, hand, xq) device tensors of the last encode's intermediates (test hook)."""
        S, ne = self.num_streams, self.ne
        xf = torch.empty((S, ne), dtype=torch.float32, device=self.device)
        eb = torch.empty((S, 64), dtype=torch.float32, device=self.device)
        hand = torch.empty((S, 8), dtype=torch.int32, device=self.device)
        xq = torch.empty((S, ne), dtype=torch.int16, device=self.device)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        rc = native.lib().lc3b_encoder_debug_read(self._h, _ptr(xf), _ptr(eb), _ptr(hand), _ptr(xq), C.c_void_p(stream))
        if rc:
            raise Lc3bError(rc, "lc3b_encoder_debug_read")
        return xf, eb, hand, xq
