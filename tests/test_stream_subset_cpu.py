"""The subset and reset entry points reject a null handle without touching a device.  Id lists that are null, out of
range, repeated or longer than the handle need a handle and are checked in test_stream_subset_gpu.py."""
import numpy as np


def test_subset_calls_reject_null_handles():
    import ctypes as C

    import lc3_codec_b200 as L
    lib = L.lib()
    ids = np.array([0], np.int32)
    p = C.c_void_p(ids.ctypes.data)
    assert lib.lc3b_decode_frames_subset(None, 16, p, 1, None, None, 150, 150, None, 480, None, None) == 2
    assert lib.lc3b_decode_frames_subset(None, 16, None, 0, None, None, 150, 150, None, 480, None, None) == 2
    assert lib.lc3b_encode_frames_subset(None, p, 1, None, 480, None, 120, 120, None) == 2
    assert lib.lc3b_encode_frames_subset(None, None, 0, None, 480, None, 120, 120, None) == 2
    for fn in (lib.lc3b_decoder_reset_streams, lib.lc3b_encoder_reset_streams):
        assert fn(None, p, 1, None) == 2
        assert fn(None, None, -1, None) == 2


def test_host_id_lists_are_int32_vectors():
    import pytest
    import torch

    from lc3_codec_b200 import Lc3bError, native
    assert native.host_ids([3, 1, 2]).tolist() == [3, 1, 2]
    assert native.host_ids(np.array([5, 0], np.int64)).dtype == np.int32
    assert native.host_ids(torch.tensor([7, 8], dtype=torch.int32)).tolist() == [7, 8]
    assert native.host_ids([]).size == 0
    for bad in ([[0, 1]], [0.5], torch.tensor([1], dtype=torch.int64), [2**31]):
        with pytest.raises(Lc3bError):
            native.host_ids(bad)
