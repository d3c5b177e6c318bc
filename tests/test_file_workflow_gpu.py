"""File-level workflows of the reference's examples (SURVEY.md 8f-2) through the C++ host mirror on the GPU:
WAV -> .lc3 (examples/encode.rs) and .lc3 -> WAV (examples/decode.rs), checked against the oracle."""
import pathlib
import struct
import subprocess

import numpy as np
import pytest

from common import assert_pcm_matches_oracle, corpus

pytestmark = pytest.mark.gpu
ROOT = pathlib.Path(__file__).resolve().parent.parent
EXE = ROOT / "examples" / "_build" / "lc3b_codec_file"


def _wav_bytes(pcm_by_channel, fs):
    nch, n = pcm_by_channel.shape
    data = np.ascontiguousarray(pcm_by_channel.T).astype("<i2").tobytes()          # interleaved
    hdr = b"RIFF" + struct.pack("<I", len(data) + 36) + b"WAVEfmt " + struct.pack("<IHHIIHH", 16, 1, nch, fs, fs * nch * 2, nch * 2, 16)
    return hdr + b"data" + struct.pack("<I", len(data)) + data


def test_wav_to_lc3_to_wav_stereo_48k(tmp_path):
    subprocess.run(["make", "-C", str(ROOT / "examples")], check=True, capture_output=True)
    F, nbytes = 30, 120
    pcm, o_frames = corpus(48000, 10, nbytes, 2, F)                  # [2, F, 480]: two channels of one file
    wav_in, lc3, wav_out = tmp_path / "in.wav", tmp_path / "x.lc3", tmp_path / "out.wav"
    wav_in.write_bytes(_wav_bytes(pcm.reshape(2, -1), 48000))
    r = subprocess.run([str(EXE), "encode", str(wav_in), str(lc3), "48000", "10", str(nbytes)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    got = np.frombuffer(lc3.read_bytes(), np.uint8).reshape(F, 2, nbytes).transpose(1, 0, 2)       # period-major file -> [ch, F, nbytes]
    assert np.array_equal(got, o_frames), "bitstream file differs from the oracle encoder"
    r = subprocess.run([str(EXE), "decode", str(lc3), str(wav_out), "48000", "10", str(nbytes), "2"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    raw = wav_out.read_bytes()
    assert raw[:4] == b"RIFF" and raw[8:16] == b"WAVEfmt " and struct.unpack("<H", raw[22:24])[0] == 2
    out = np.frombuffer(raw[44:], "<i2").reshape(F * 480, 2).T.reshape(2, F, 480)
    assert_pcm_matches_oracle(out, 48000, 10, o_frames)
