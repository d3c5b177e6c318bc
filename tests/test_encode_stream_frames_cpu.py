"""The time-parallel encode entry points reject null handles and pointers without touching a device."""
import ctypes as C


def test_encode_stream_frames_rejects_null_handles_and_pointers():
    import lc3_codec_b200 as L
    lib = L.lib()
    n = C.c_size_t(0)
    assert lib.lc3b_encoder_multi_scratch_bytes(None, 4, C.byref(n)) == 2
    assert lib.lc3b_encoder_multi_scratch_bytes(None, 4, None) == 2
    assert lib.lc3b_encode_stream_frames(None, None, 4, None, 120, 120, None, 1 << 20, None) == 2
