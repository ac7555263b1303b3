"""CPU tests of the native FLAC reader (csrc/flac.cpp behind tw_flac_decode; SURVEY.md §8f rank 2) against streams
written by the test-side encoder (tests/flac_writer.py): bit-exact PCM for every subframe type, Rice variant, stereo
mode, bit depth and block-size / sample-rate coding the format has, ragged last blocks, unknown stream length, an ID3
prefix, trailing garbage; corrupted bytes are rejected through the frame CRCs and the STREAMINFO MD5."""
import ctypes as C

import numpy as np
import pytest

import flac_writer as W
from turbo_whisper_workspace_b200 import _lib
from turbo_whisper_workspace_b200.pipeline import _read_flac, ffmpeg_read


def _signal(rng, n, ch, bps, kind):
    lim = 1 << (bps - 1)
    t = np.arange(n)
    if kind == "noise":
        x = rng.integers(-lim, lim, size=(n, ch))
    elif kind == "tone":
        x = np.stack([0.6 * lim * np.sin(2 * np.pi * (0.01 + 0.003 * c) * t + c) for c in range(ch)], 1) \
            + rng.integers(-3, 4, size=(n, ch))
    elif kind == "steps":      # constant runs (CONSTANT subframes) and values with trailing zero bits (wasted bits)
        x = (np.repeat(rng.integers(-lim // 8, lim // 8, size=(n // 64 + 1, ch)), 64, axis=0)[:n] // 8) * 8
    elif kind == "silence":
        x = np.zeros((n, ch))
    else:                      # correlated stereo
        base = 0.5 * lim * np.sin(2 * np.pi * 0.004 * t)
        x = np.stack([base + rng.integers(-20, 21, size=n) for _ in range(ch)], 1)
    return np.clip(np.round(x), -lim, lim - 1).astype(np.int64)


def _decode(payload):
    lib = _lib.load()
    buf = np.frombuffer(payload, dtype=np.uint8)
    info = _lib.FlacInfo()
    assert lib.tw_flac_info_read(buf.ctypes.data_as(C.c_void_p), len(payload), C.byref(info)) == 0
    n = C.c_int64(0)
    assert lib.tw_flac_decode(buf.ctypes.data_as(C.c_void_p), len(payload), None, 0, C.byref(n)) == 0
    out = np.empty((n.value, info.channels), dtype=np.int32)
    rc = lib.tw_flac_decode(buf.ctypes.data_as(C.c_void_p), len(payload), out.ctypes.data_as(C.c_void_p), n.value, C.byref(n))
    assert rc == 0, lib.tw_last_error()
    return info, out


@pytest.mark.parametrize("bps", [8, 12, 16, 20, 24])
def test_round_trip_all_coding_tools(bps):
    rng = np.random.default_rng(bps)
    case = 0
    for ch in (1, 2, 3):
        for kind in ("noise", "tone", "steps", "silence", "stereo"):
            for blocksize in (16, 192, 1000, 4096):
                n = int(rng.integers(1, 3 * blocksize + 2))
                sr = [8000, 16000, 22050, 44100, 48000, 96000, 192000, 12345, 700001][case % 9]
                pcm = _signal(rng, n, ch, bps, kind)
                payload = W.encode(pcm, sr, bps, seed=case, blocksize=blocksize, total_known=case % 3 != 0,
                                   with_md5=case % 4 != 0, id3=case % 7 == 0)
                info, out = _decode(payload)
                assert (info.sample_rate, info.channels, info.bits_per_sample) == (sr, ch, bps)
                assert out.shape == pcm.shape and (out == pcm).all(), (case, ch, kind, blocksize)
                got = _read_flac(payload)          # python wrapper incl. the MD5 check and the dtype contract
                assert got[1] == sr
                if bps == 16:
                    assert got[0].dtype == np.int16 and (got[0] == pcm).all()
                else:
                    np.testing.assert_array_equal(got[0], (pcm / float(1 << (bps - 1))).astype(np.float32))
                case += 1
    assert case == 60


def test_many_small_frames_multibyte_frame_numbers_and_trailing_bytes():
    rng = np.random.default_rng(1)
    pcm = _signal(rng, 16 * 2500 + 5, 2, 16, "tone")      # 2501 frames: frame numbers need 1, 2 and 3 coded bytes
    payload = W.encode(pcm, 16000, 16, seed=3, blocksize=16) + b"TAG" + bytes(125)   # ID3v1-style trailer
    info, out = _decode(payload)
    assert (out == pcm).all()
    # through the pipeline's reader at the target rate: mono down-mix on the host
    x = ffmpeg_read(payload, 16000)
    np.testing.assert_allclose(x, (pcm.astype(np.float32) / 32768.0).mean(axis=1), rtol=0, atol=1e-7)


def test_corruption_is_detected():
    lib = _lib.load()
    rng = np.random.default_rng(2)
    pcm = _signal(rng, 5000, 2, 16, "tone")
    payload = bytearray(W.encode(pcm, 44100, 16, seed=5, blocksize=1152))
    first_frame = payload.index(b"\xff\xf8", 42)
    hits = 0
    for off in (first_frame + 2, first_frame + 40, len(payload) // 2, len(payload) - 3):
        bad = bytearray(payload)
        bad[off] ^= 0x10
        with pytest.raises(ValueError):
            _read_flac(bytes(bad))
        hits += 1
    assert hits == 4
    # a wrong MD5 signature with intact frames
    bad = bytearray(payload)
    bad[4 + 4 + 18] ^= 0xff
    with pytest.raises(ValueError, match="MD5"):
        _read_flac(bytes(bad))
    assert _read_flac(bytes(bad), verify_md5=False)[0].shape == (5000, 2)
    # truncated stream, not a FLAC stream, null arguments
    with pytest.raises(ValueError):
        _read_flac(bytes(payload[:len(payload) // 2]))
    assert _read_flac(b"RIFF....WAVE") is None
    n = C.c_int64(0)
    assert lib.tw_flac_decode(None, 0, None, 0, C.byref(n)) != 0 and b"tw_flac_decode" in lib.tw_last_error()
    buf = np.frombuffer(b"fLaCxxxx", dtype=np.uint8)
    assert lib.tw_flac_decode(buf.ctypes.data_as(C.c_void_p), 8, None, 0, C.byref(n)) != 0
