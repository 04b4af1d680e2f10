"""CPU tests of the checker for the file formats either side of the path (SURVEY 8f-4): the C restatement of the
.flan sample codec against the reference's own PVBuffer::save / load (compiled verbatim), byte for byte; the WAV
PCM-24 restatement (libsndfile is absent: parity unpinned) against Python's stdlib `wave` reader and known answers."""
import os
import struct

import numpy as np
import pytest

from reference_records import Records, file_codec_reference


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def pv_fixture(seed=3, C=2, F=9, B=65, sr=44100.0):
    rng = np.random.default_rng(seed)
    pv = np.empty((C, F, B, 2), np.float32)
    pv[..., 0] = rng.uniform(0, 40, (C, F, B))
    pv[..., 1] = rng.uniform(-100, sr / 2, (C, F, B))
    # edge cases of the clamp / truncation: exactly the limits, beyond them, tiny and negative values
    pv[0, 0, :8, 0] = [0.0, 128.0, 127.99999, 1e-6, -3.0, 500.0, 64.0, 1.0 / 65536]
    pv[0, 0, :6, 1] = [sr, -sr, sr * 2, 0.0, -0.004, 22050.0]
    return pv, sr


@pytest.fixture(scope="module")
def rec():
    r = Records("test_oracle_io")
    yield r
    r.save()


def test_flan_codec_matches_reference_file_bytes(oracle, rec, tmp_path):
    pv, sr = pv_fixture()
    ar, W = oracle.analysis_rate(sr, 32), 128
    ref = file_codec_reference()
    if ref is not None:
        path = str(tmp_path / "ref.flan")
        ref.save_flan(path, pv, sr, ar, W)
        raw = np.fromfile(path, np.uint8)
        got, sr2, ar2, W2 = ref.load_flan(path)
        header = np.array([sr2, ar2, W2], np.float64)
        rec.check("save.file", raw, raw, whole=True)
        rec.check("load.header", header, header)
    else:           # what the reference's save wrote and its load returned, as stored
        raw = rec.stored_array("save.file")
        sr2, ar2, W2 = rec.stored_array("load.header").tolist()
        got = None
    assert raw[:4].tobytes() == b"RIFF" and raw[8:12].tobytes() == b"PV\0\0" and raw[12:16].tobytes() == b"fmt "
    fmt = struct.unpack("<IHHIIIIIIH", raw[16:50].tobytes())
    assert fmt == (30, 1, 2, 9, 65, 44100, 32, 128, 24, 1)
    assert raw[50:54].tobytes() == b"data" and struct.unpack("<I", raw[54:58].tobytes())[0] == pv.size * 3
    assert np.array_equal(raw[58:], oracle.flan_encode(pv, sr))
    # ... and back: the reference's load against the restated decode, bit for bit; load keeps the hop as analysis rate
    assert (sr2, ar2, W2) == (44100.0, 32.0, 128)
    decoded = oracle.flan_decode(raw[58:], pv.shape[:3], sr)
    rec.check("load.pv", decoded, got)
    got = decoded
    # quantisation error bound away from the clamp: 2^-23 of full scale
    inside = (np.abs(pv[..., 0]) < 128) & (np.abs(pv[..., 1]) < sr)
    assert np.max(np.abs(got[..., 0] - pv[..., 0])[inside]) <= 128 * 2.0 ** -23 * 1.0001
    assert np.max(np.abs(got[..., 1] - pv[..., 1])[inside]) <= sr * 2.0 ** -23 * 1.0001


def test_flan_codec_known_answers(oracle):
    sr = 48000.0
    pv = np.zeros((1, 1, 3, 2), np.float32)        # dft size 4
    pv[0, 0, :, 0] = [4.0, -4.0, 2.0]              # +1 -> 0x800000 (wraps to -1 on load, as in the reference), -1, 0.5
    pv[0, 0, :, 1] = [24000.0, 0.0, -12000.0]
    b = oracle.flan_encode(pv, sr).reshape(-1, 3)
    assert b.tolist() == [[0, 0, 0x80], [0, 0, 0x40], [0, 0, 0x80], [0, 0, 0], [0, 0, 0x40], [0, 0, 0xE0]]
    back = oracle.flan_decode(b.reshape(-1), (1, 1, 3), sr)
    assert back[0, 0, :, 0].tolist() == [-4.0, -4.0, 2.0] and back[0, 0, :, 1].tolist() == [24000.0, 0.0, -12000.0]


def test_pcm24_restatement_against_stdlib_wave_and_known_answers(oracle, tmp_path):
    import wave
    rng = np.random.default_rng(4)
    x = rng.uniform(-1.2, 1.2, (2, 1001)).astype(np.float32)
    x[0, :6] = [0.0, 1.0, -1.0, 0.5, 2.0 ** -24, -2.0 ** -23]
    b = oracle.pcm24_encode(x)
    q = b.reshape(-1, 3).astype(np.int32)
    v = ((q[:, 0] | (q[:, 1] << 8) | (q[:, 2] << 16)) << 8) >> 8
    v = v.reshape(1001, 2).T                                  # frames interleaved
    want = np.rint(np.clip(x, -1, 1).astype(np.float32) * np.float32(8388607.0)).astype(np.int32)
    assert np.array_equal(v, want)
    assert v[0, :5].tolist() == [0, 8388607, -8388607, 4194304, 0]      # 4194303.5 and 0.5 round to even
    path = str(tmp_path / "a.wav")
    with wave.open(path, "wb") as w:
        w.setnchannels(2); w.setsampwidth(3); w.setframerate(44100); w.writeframes(b.tobytes())
    with wave.open(path, "rb") as w:
        assert (w.getnchannels(), w.getsampwidth(), w.getnframes()) == (2, 3, 1001)
        assert w.readframes(1001) == b.tobytes()
    back = oracle.pcm24_decode(b, 2, 1001)
    assert np.array_equal(back, (want / np.float32(8388608.0)).astype(np.float32))
