"""The ragged time-parallel entry points reject a null handle without touching a device, and host frame-count lists
convert like id lists.  Everything that needs a handle is in test_ragged_stream_frames_gpu.py."""
import ctypes as C

import numpy as np


def test_ragged_calls_reject_null_handles():
    import lc3_codec_b200 as L
    lib = L.lib()
    ids = np.array([0], np.int32)
    counts = np.array([2], np.int32)
    pi, pc = C.c_void_p(ids.ctypes.data), C.c_void_p(counts.ctypes.data)
    n = C.c_size_t(0)
    assert lib.lc3b_decoder_multi_subset_scratch_bytes(None, 1, 2, C.byref(n)) == 2
    assert lib.lc3b_encoder_multi_subset_scratch_bytes(None, 1, 2, C.byref(n)) == 2
    assert lib.lc3b_decode_stream_frames_subset(None, 16, pi, pc, 1, None, None, 150, 150, None, None, None, 0, None) == 2
    assert lib.lc3b_decode_stream_frames_subset(None, 16, None, None, 0, None, None, 150, 150, None, None, None, 0, None) == 2
    assert lib.lc3b_encode_stream_frames_subset(None, pi, pc, 1, None, None, 120, 120, None, 0, None) == 2
    assert lib.lc3b_encode_stream_frames_subset(None, None, None, 0, None, None, 120, 120, None, 0, None) == 2


def test_host_counts_are_int32_vectors_matching_the_ids():
    import pytest
    import torch

    from lc3_codec_b200 import Lc3bError, native
    assert native.host_counts([3, 0, 200], 3).tolist() == [3, 0, 200]
    assert native.host_counts(np.array([5, 1], np.int64), 2).dtype == np.int32
    assert native.host_counts(torch.tensor([7, 8], dtype=torch.int32), 2).tolist() == [7, 8]
    assert native.host_counts([], 0).size == 0
    assert native.host_counts([-1], 1).tolist() == [-1]             # signs are the library's to check
    for bad, n in (([[0, 1]], 1), ([0.5], 1), (torch.tensor([1], dtype=torch.int64), 1), ([2**31], 1), ([1, 2], 3)):
        with pytest.raises(Lc3bError):
            native.host_counts(bad, n)
