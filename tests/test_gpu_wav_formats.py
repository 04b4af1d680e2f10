"""GPU tests of WAV files of every sample type libsndfile writes for SF_FORMAT_WAV (PCM_U8, PCM_16, PCM_24, PCM_32, FLOAT,
DOUBLE) through the C ABI, the C++ API and the example program: the device codecs byte- and bit-exact against the
oracle's restatement (tests/test_oracle_wav_formats.py pins that restatement), files the engine writes as scipy and
stdlib `wave` read them, files written elsewhere, streaming over several chunks, and refusals."""
import ctypes
import hashlib
import os
import struct
import subprocess
import wave

import numpy as np
import pytest

from flan_b200 import capi
from flan_b200.signals import noise_chirp
from wav_files import (ALL, DOUBLE, FLOAT, NAME, PCM_16, PCM_24, PCM_32, PCM_U8, WIDTH, OracleWav, build_wav, chunk,
                       data_bytes, fmt_fields, interleave)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def oracle(oracle):
    """The checker's WAV sample codecs (tests/cpp/wav_oracle.c), next to the session's oracle library."""
    return OracleWav(oracle)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.fixture(scope="module")
def eng():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from flan_b200.engine import Engine
    return Engine(0)


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def signal(C, n, seed):
    """Uniform noise past full scale, with the values the write rules treat specially at the start."""
    rng = np.random.default_rng(seed)
    x = rng.uniform(-1.2, 1.2, (C, n)).astype(np.float32)
    special = np.array([1.0, -1.0, 0.0, -0.0, np.inf, -np.inf, 0.5, -0.5, 2.0 ** -32, 3 * 2.0 ** -32, 5 * 2.0 ** -32,
                        2.0 ** -149, 1 - 2.0 ** -24, 1.5, np.nan], np.float32)
    k = min(n, special.size)
    x[0, :k] = special[:k]
    if C > 1:
        x[C - 1, -k:] = special[:k][::-1]
    return x


def decode_input(oracle, t, C, n, seed):
    """Bytes to decode: every bit pattern at random (for DOUBLE mostly NaNs and huge values, so half of them are samples
    in [-1, 1] and rounding, overflow and underflow cases instead)."""
    rng = np.random.default_rng(seed)
    b = rng.integers(0, 256, C * n * WIDTH[t], dtype=np.uint8)
    if t == DOUBLE:
        d = b.view("<f8").copy()
        d[::2] = rng.uniform(-1, 1, d[::2].size)
        edge = np.array([1 + 2.0 ** -24, 1 + 3 * 2.0 ** -24, 1e300, -1e300, 1e-50, 2.0 ** -150, 3 * 2.0 ** -150, -0.0,
                         np.inf, 3.4028235677973366e38, 2.0 ** -126 * (1 - 2.0 ** -25)])
        d[:min(d.size, edge.size)] = edge[:min(d.size, edge.size)]
        b = d.view(np.uint8)
    return b


@pytest.mark.parametrize("n", [1, 4095, 4096 * 3 + 1, 100003])
@pytest.mark.parametrize("C", [1, 2, 3, 8])
@pytest.mark.parametrize("t", ALL, ids=lambda t: NAME[t])
def test_codec_byte_exact(eng, oracle, t, C, n):
    x = signal(C, n, seed=C * 7 + n)
    x[0, :n // 3:7] = np.array([0x7FC00001, 0xFFC12345, 0x7F800001], np.uint32).view(np.float32)[np.arange(x[0, :n // 3:7].size) % 3]
    want = oracle.pcm_encode(x, t)
    assert np.array_equal(eng.pcm_encode(dev(x), t).cpu().numpy(), want)
    b = decode_input(oracle, t, C, n, seed=n + t)
    assert np.array_equal(bits(eng.pcm_decode(dev(b), C, n, t).cpu().numpy()), bits(oracle.pcm_decode(b, C, n, t)))
    back = eng.pcm_decode(dev(want), C, n, t).cpu().numpy()
    assert np.array_equal(bits(back), bits(oracle.pcm_decode(want, C, n, t)))


def test_known_answers_and_pcm24_entry_points(eng, oracle):
    x = np.array([[1.0, -1.0, np.nan, 0.5, -0.0, 2.0, -np.inf, 2.0 ** -32]], np.float32)
    b = eng.pcm_encode(dev(x), PCM_32).cpu().numpy().view("<u4")
    assert list(b) == [0x80000000, 0x80000000, 0x80000000, 0x40000000, 0, 0x80000000, 0x80000000, 0]
    assert list(eng.pcm_encode(dev(x), PCM_U8).cpu().numpy()) == [255, 1, 128, 192, 128, 255, 1, 128]
    assert list(eng.pcm_encode(dev(x), PCM_16).cpu().numpy().view("<i2")) == [32767, -32767, 0, 16384, 0, 32767, -32767, 0]
    f = eng.pcm_encode(dev(x), FLOAT).cpu().numpy().view("<u4")
    assert f[2] == x.view(np.uint32)[0, 2] and f[4] == 0x80000000 and f[5] == 0x3F800000
    d = eng.pcm_encode(dev(x), DOUBLE).cpu().numpy().view("<f8")
    assert np.isnan(d[2]) and d[0] == 1.0 and d[5] == 1.0 and np.signbit(d[4])
    # FLOAT keeps NaN payloads, signalling ones too; DOUBLE converts them as x86 does (quiet bit set, payload kept)
    nans = np.array([[0x7FC00001, 0xFFC12345, 0x7F800001, 0xFFBFFFFF]], np.uint32).view(np.float32)
    assert np.array_equal(eng.pcm_encode(dev(nans), FLOAT).cpu().numpy().view("<u4"), nans.view(np.uint32)[0])
    assert np.array_equal(eng.pcm_encode(dev(nans), DOUBLE).cpu().numpy().view("<u8"), nans.astype(np.float64).view(np.uint64)[0])
    back = eng.pcm_decode(eng.pcm_encode(dev(nans), DOUBLE), 1, 4, DOUBLE).cpu().numpy()
    assert np.array_equal(bits(back)[0], nans.view(np.uint32)[0] | 0x00400000)
    # the PCM_24 forms are the general codec's PCM_24
    y = signal(3, 5001, 9)
    assert np.array_equal(eng.pcm24_encode(dev(y)).cpu().numpy(), eng.pcm_encode(dev(y), PCM_24).cpu().numpy())
    raw = eng.pcm_encode(dev(y), PCM_24)
    assert np.array_equal(bits(eng.pcm24_decode(raw, 3, 5001).cpu().numpy()), bits(eng.pcm_decode(raw, 3, 5001, PCM_24).cpu().numpy()))
    with pytest.raises(capi.FlanB200Error) as e:
        eng.ctx.call("flan_b200_pcm_encode", eng._chk(dev(y)), 3, 5001, 1, eng._chk(raw, raw.dtype))     # PCM_S8
    assert e.value.code == capi.INVALID


SCIPY_DTYPE = {PCM_U8: np.uint8, PCM_16: np.int16, PCM_32: np.int32, FLOAT: np.float32, DOUBLE: np.float64}
FILE_DTYPE = {PCM_U8: "u1", PCM_16: "<i2", PCM_32: "<i4", FLOAT: "<f4", DOUBLE: "<f8"}


@pytest.mark.parametrize("t", ALL, ids=lambda t: NAME[t])
def test_engine_files_read_by_scipy_and_wave(eng, oracle, tmp_path, t):
    from scipy.io import wavfile
    C, n, sr = 3, 20001, 44100.0
    x = signal(C, n, seed=t)
    path = str(tmp_path / ("%s.wav" % NAME[t]))
    eng.save_wav(path, dev(x), sr, t)
    want = oracle.pcm_encode(x, t)
    raw = open(path, "rb").read()
    tag, ch, rate, byte_rate, block, nbits = fmt_fields(raw)
    ieee = t in (FLOAT, DOUBLE)
    assert (tag, ch, rate, byte_rate, block, nbits) == (3 if ieee else 1, C, 44100, 44100 * C * WIDTH[t], C * WIDTH[t], 8 * WIDTH[t])
    assert len(chunk(raw, b"fmt ")) == (18 if ieee else 16)
    if ieee:
        assert struct.unpack("<I", chunk(raw, b"fact"))[0] == n
    else:
        assert chunk(raw, b"fact") is None and len(raw) - len(want) - (len(want) & 1) == 44
    assert struct.unpack("<I", raw[4:8])[0] == len(raw) - 8
    assert np.array_equal(data_bytes(path), want)
    assert eng.wav_format(path) == t
    rate2, v = wavfile.read(path)
    assert rate2 == 44100 and v.shape == (n, C)
    if t == PCM_24:         # scipy returns 24-bit samples left-justified in int32
        b = want.reshape(n, C, 3).astype(np.int64)
        ints = ((b[..., 0] | (b[..., 1] << 8) | (b[..., 2] << 16)) << 40) >> 40
        assert np.array_equal(v.astype(np.int64), ints << 8)
    else:
        assert v.dtype == np.dtype(FILE_DTYPE[t]) and np.array_equal(v.view(np.uint8).reshape(-1), want)
    if not ieee:
        with wave.open(path, "rb") as w:
            assert (w.getnchannels(), w.getsampwidth(), w.getframerate(), w.getnframes()) == (C, WIDTH[t], 44100, n)
            assert w.readframes(n) == want.tobytes()
    y, sr2 = eng.load_wav(path)
    assert sr2 == sr
    assert np.array_equal(bits(y.cpu().numpy()), bits(oracle.pcm_decode(want, C, n, t)))


@pytest.mark.parametrize("t", [PCM_U8, PCM_16, PCM_32, FLOAT, DOUBLE], ids=lambda t: NAME[t])
def test_scipy_files_load_bit_exact(eng, oracle, tmp_path, t):
    from scipy.io import wavfile
    C, n = 2, 30001
    rng = np.random.default_rng(t)
    dt = SCIPY_DTYPE[t]
    if np.issubdtype(dt, np.integer):
        info = np.iinfo(dt)
        v = rng.integers(info.min, int(info.max) + 1, (n, C), dtype=np.int64).astype(dt)
    else:
        v = rng.uniform(-1.5, 1.5, (n, C)).astype(dt)
    path = str(tmp_path / "s.wav")
    wavfile.write(path, 22050, v)
    assert eng.wav_format(path) == t
    y, sr = eng.load_wav(path)
    assert sr == 22050.0 and tuple(y.shape) == (C, n)
    assert np.array_equal(bits(y.cpu().numpy()), bits(oracle.pcm_decode(data_bytes(path), C, n, t)))


def write(tmp_path, name, raw):
    path = str(tmp_path / name)
    with open(path, "wb") as f:
        f.write(raw)
    return path


HAND_BUILT = [
    # name, C, subtype, build_wav keywords
    ("ext_pcm24_3ch", 3, PCM_24, dict(tag=1, bits=24, extensible=True)),
    ("ext_float_6ch", 6, FLOAT, dict(tag=3, bits=32, extensible=True)),
    ("ext_20_in_3", 2, PCM_24, dict(tag=1, bits=24, extensible=True, valid_bits=20)),
    ("plain_20_in_3", 2, PCM_24, dict(tag=1, bits=20, block=6)),
    ("list_before_data", 2, PCM_16, dict(tag=1, bits=16, before_data=[(b"LIST", b"INFOISFT\x05\x00\x00\x00test\x00\x00")])),
    ("odd_chunk", 1, PCM_U8, dict(tag=1, bits=8, before_data=[(b"junk", b"abcde"), (b"PEAK", bytes(24))])),
    ("ext_double", 1, DOUBLE, dict(tag=3, bits=64, extensible=True, before_data=[(b"fact", struct.pack("<I", 999))])),
]


@pytest.mark.parametrize("name,C,t,kw", HAND_BUILT, ids=[h[0] for h in HAND_BUILT])
def test_hand_built_files_load_bit_exact(eng, oracle, tmp_path, name, C, t, kw):
    n = 999                                        # odd: with one channel of U8 the data chunk has a pad byte
    x = signal(C, n, seed=len(name))
    data = oracle.pcm_encode(x, t)
    path = write(tmp_path, name + ".wav", build_wav(data, C, 32000, **kw))
    assert eng.wav_format(path) == t
    y, sr = eng.load_wav(path)
    assert sr == 32000.0 and tuple(y.shape) == (C, n)
    assert np.array_equal(bits(y.cpu().numpy()), bits(oracle.pcm_decode(data, C, n, t)))


REFUSED = [
    ("adpcm", dict(tag=2, bits=4, block=256)),
    ("alaw", dict(tag=6, bits=8)),
    ("mulaw", dict(tag=7, bits=8)),
    ("block_align", dict(tag=1, bits=16, block=3)),
    ("bits_vs_container", dict(tag=1, bits=24, block=4)),
    ("float_16", dict(tag=3, bits=16)),
    ("ext_other_guid", dict(tag=1, bits=16, extensible=True, sub_tail=bytes(14))),
]


@pytest.mark.parametrize("name,kw", REFUSED, ids=[r[0] for r in REFUSED])
def test_other_formats_are_unsupported(eng, tmp_path, name, kw):
    import torch
    path = write(tmp_path, name + ".wav", build_wav(bytes(64), 1, 8000, **kw))
    for call in (lambda: eng.wav_format(path), lambda: eng.load_wav(path)):
        with pytest.raises(capi.FlanB200Error) as e:
            call()
        assert e.value.code == capi.UNSUPPORTED
        assert "tag %d" % (0xFFFE if kw.get("extensible") else kw["tag"]) in str(e.value)
    out = torch.zeros(64, dtype=torch.float32, device="cuda")
    with pytest.raises(capi.FlanB200Error) as e:
        eng.ctx.call("flan_b200_load_wav", path.encode(), eng._chk(out), 64)
    assert e.value.code == capi.UNSUPPORTED


@pytest.mark.parametrize("t", ALL, ids=lambda t: NAME[t])
def test_saves_over_4_gib_are_refused_before_the_file_exists(eng, tmp_path, t):
    x = dev(np.zeros((2, 16), np.float32))
    header = 58 if t in (FLOAT, DOUBLE) else 44
    n = (0xFFFFFFFF - (header - 8)) // (2 * WIDTH[t]) + 1
    path = str(tmp_path / "big.wav")
    eng._bind_stream()
    with pytest.raises(capi.FlanB200Error) as e:
        eng.ctx.call("flan_b200_save_wav_as", path.encode(), eng._chk(x), 2, n, 48000.0, t)
    assert e.value.code == capi.UNSUPPORTED
    assert not os.path.exists(path)


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).view(np.uint8)).hexdigest()


@pytest.mark.parametrize("C,n,t", [(2, 30_000_000, DOUBLE), (3, 25_000_000, PCM_24), (3, 9_000_001, PCM_U8)],
                         ids=["double_2ch", "pcm24_3ch", "u8_3ch"])
def test_streaming_over_several_chunks(eng, oracle, tmp_path, C, n, t):
    # chunks hold about 192 MiB of file in whole multiples of 4096 frames: these files take 2 or 3 of them
    frames_per_chunk = (192 << 20) // WIDTH[t] // C // 4096 * 4096
    assert n > frames_per_chunk or t == PCM_U8
    rng = np.random.default_rng(n)
    x = rng.uniform(-1.1, 1.1, (C, n)).astype(np.float32)
    path = str(tmp_path / "long.wav")
    eng.save_wav(path, dev(x), 48000.0, t)
    want = oracle.pcm_encode(x, t)
    assert sha(data_bytes(path)) == sha(want)
    y, _ = eng.load_wav(path)
    assert sha(bits(y.cpu().numpy())) == sha(bits(oracle.pcm_decode(want, C, n, t)))


# ---- the C++ API ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def drv(eng):
    from flan_b200 import build
    build.build_host()
    L = ctypes.CDLL(build.wav_test_path())
    fp = ctypes.POINTER(ctypes.c_float)
    L.api_wav_save.argtypes = [fp, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_char_p, ctypes.c_int]
    L.api_wav_load.argtypes = [ctypes.c_char_p, fp, ctypes.c_int64, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_float)]
    return L


def fptr(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))


@pytest.mark.parametrize("t", [PCM_16, FLOAT], ids=lambda t: NAME[t])
def test_cpp_audio_load_of_16_bit_and_float_files(drv, oracle, tmp_path, t):
    from scipy.io import wavfile
    C, n = 2, 12345
    rng = np.random.default_rng(t)
    v = rng.integers(-32768, 32768, (n, C)).astype(np.int16) if t == PCM_16 else rng.uniform(-1, 1, (n, C)).astype(np.float32)
    path = str(tmp_path / "in.wav")
    wavfile.write(path, 44100, v)
    out = np.zeros((C, n), np.float32)
    ch, sr = ctypes.c_int(), ctypes.c_float()
    assert drv.api_wav_load(path.encode(), fptr(out), out.size, ctypes.byref(ch), ctypes.byref(sr)) == n
    assert (ch.value, sr.value) == (C, 44100.0)
    assert np.array_equal(bits(out), bits(oracle.pcm_decode(data_bytes(path), C, n, t)))


# which (tests/cpp/wav_formats_driver.cpp) -> the sample type written
CPP_SAVES = [(0, PCM_24), (1, FLOAT), (2, PCM_16), (3, PCM_24), (7, PCM_U8), (8, PCM_32), (9, DOUBLE)]


@pytest.mark.parametrize("which,t", CPP_SAVES, ids=["default", "float", "pcm16", "pcm24", "u8_little", "pcm32_file", "double"])
def test_cpp_audio_save_formats(drv, oracle, tmp_path, which, t):
    C, n = 2, 7001
    x = np.stack([noise_chirp(n, 44100.0, 1), noise_chirp(n, 44100.0, 2) * np.float32(2.0)])      # second channel clips
    path = str(tmp_path / "out.wav")
    assert drv.api_wav_save(fptr(x), C, n, 44100.0, path.encode(), which) == 1
    raw = open(path, "rb").read()
    assert fmt_fields(raw)[0] == (3 if t in (FLOAT, DOUBLE) else 1) and fmt_fields(raw)[5] == 8 * WIDTH[t]
    assert np.array_equal(data_bytes(path), oracle.pcm_encode(x, t))


@pytest.mark.parametrize("which", [4, 5, 6], ids=["aiff", "pcm_s8", "big_endian"])
def test_cpp_audio_save_refuses_other_formats(drv, tmp_path, capfd, which):
    x = np.zeros((1, 100), np.float32)
    path = str(tmp_path / "no.wav")
    capfd.readouterr()
    assert drv.api_wav_save(fptr(x), 1, 100, 48000.0, path.encode(), which) == 0
    assert "Sound file formatting invalid while attempting to save to " + path in capfd.readouterr().out
    assert not os.path.exists(path)


def test_example_program_reads_a_16_bit_file(eng, tmp_path):
    from flan_b200 import build
    build.build_host()
    exe = os.path.join(os.path.dirname(build.host_path()), "pv_chain")
    sr, n = 44100, 44100 * 2
    x = np.stack([noise_chirp(n, float(sr), 5), noise_chirp(n, float(sr), 6)]) * np.float32(0.5)
    src, out = str(tmp_path / "in16.wav"), str(tmp_path / "out.wav")
    with wave.open(src, "wb") as w:
        w.setnchannels(2)
        w.setsampwidth(2)
        w.setframerate(sr)
        w.writeframes(interleave(np.rint(x * 32767).astype("<i2")).tobytes())
    r = subprocess.run([exe, src, out, "1.5", "2.0"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    with wave.open(out, "rb") as w:
        assert (w.getnchannels(), w.getsampwidth(), w.getframerate()) == (2, 3, sr)
        frames = w.getnframes()
        raw = np.frombuffer(w.readframes(frames), np.uint8).reshape(-1, 3).astype(np.int32)
    assert abs(frames - 2 * n) <= 2 * 4096
    v = ((raw[:, 0] | (raw[:, 1] << 8) | (raw[:, 2] << 16)) << 8) >> 8
    assert np.sqrt(np.mean((v / 8388608.0) ** 2)) > 0.01
