"""CPU tests of the checker's WAV sample codecs (tests/cpp/wav_oracle.c wavo_pcm_encode / wavo_pcm_decode). libsndfile,
whose default conversions they restate, is not available, so parity with it stays unpinned; the restatement is pinned here
to numpy float32 arithmetic, exhaustively where the codes are few, to known answers, to files that scipy and Python's
stdlib `wave` write, and for PCM_24 to the oracle's own restatement (oracle/pv_oracle.c pvo_pcm24_*)."""
import wave

import numpy as np
import pytest

from wav_files import ALL, DOUBLE, FLOAT, PCM_16, PCM_24, PCM_32, PCM_U8, WIDTH, OracleWav, data_bytes

F32 = np.float32


@pytest.fixture(scope="module")
def oracle(oracle):
    """The checker's WAV sample codecs (tests/cpp/wav_oracle.c), next to the session's oracle library."""
    return OracleWav(oracle)


def bits32(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def test_widths_and_unknown_codes(oracle):
    for t in ALL:
        assert oracle.pcm_width(t) == WIDTH[t]
    for t in (0, 1, 8, 0x10, -1):          # PCM_S8 (1) is not a WAV sub-type
        assert oracle.pcm_width(t) == 0


def test_pcm24_is_the_oracles_pcm24_restatement(oracle):
    rng = np.random.default_rng(24)
    x = rng.uniform(-1.2, 1.2, (3, 4099)).astype(np.float32)
    x[0, :8] = [1.0, -1.0, 0.0, -0.0, np.nan, np.inf, -np.inf, 0.5]
    b = oracle.pcm_encode(x, PCM_24)
    assert np.array_equal(b, oracle.base.pcm24_encode(x))
    r = rng.integers(0, 256, 3 * 4099 * 3, dtype=np.uint8)
    assert np.array_equal(bits32(oracle.pcm_decode(r, 3, 4099, PCM_24)), bits32(oracle.base.pcm24_decode(r, 3, 4099)))


def test_u8_decode_every_code(oracle):
    codes = np.arange(256, dtype=np.uint8)
    got = oracle.pcm_decode(codes, 1, 256, PCM_U8)[0]
    want = (codes.astype(np.int32) - 128).astype(F32) * F32(1.0 / 0x80)
    assert np.array_equal(bits32(got), bits32(want))
    assert got[0] == -1.0 and got[128] == 0.0 and got[255] == F32(127 / 128)


def test_pcm16_decode_every_code(oracle):
    v = np.arange(-32768, 32768, dtype=np.int32).astype("<i2")
    got = oracle.pcm_decode(v.view(np.uint8), 1, v.size, PCM_16)[0]
    want = v.astype(F32) * F32(1.0 / 0x8000)
    assert np.array_equal(bits32(got), bits32(want))


def test_pcm32_decode_rounds_to_nearest_even(oracle):
    edge = [-2 ** 31, 2 ** 31 - 1, 0, 1, -1, 2 ** 24 - 1, 2 ** 24, 2 ** 24 + 1, 2 ** 24 + 2, 2 ** 24 + 3,
            -(2 ** 24 + 1), -(2 ** 24 + 3), 2 ** 25 + 2, 2 ** 25 + 6, 2 ** 30 + 64, 2 ** 31 - 128, 2 ** 31 - 64]
    rng = np.random.default_rng(32)
    v = np.concatenate([np.array(edge, np.int64), rng.integers(-2 ** 31, 2 ** 31, 20000)]).astype("<i4")
    got = oracle.pcm_decode(v.view(np.uint8), 1, v.size, PCM_32)[0]
    want = v.astype(F32) * F32(2.0 ** -31)              # numpy's int -> float32 rounds to nearest even
    assert np.array_equal(bits32(got), bits32(want))
    assert got[0] == -1.0 and got[1] == 1.0             # INT_MAX reads as full scale
    assert got[7] == F32(2 ** 24) * F32(2.0 ** -31)     # 2^24 + 1 ties to the even 2^24
    assert got[9] == F32(2 ** 24 + 4) * F32(2.0 ** -31)


def test_float_bits_pass_both_ways(oracle):
    pats = np.array([0x00000000, 0x80000000, 0x3F800000, 0xBF800000, 0x00000001, 0x807FFFFF, 0x00400000,
                     0x7F800000, 0xFF800000, 0x7FC00000, 0x7FC00001, 0xFFC12345, 0x7F800001, 0xFFBFFFFF, 0x3F7FFFFF,
                     0x3F800001, 0x7F7FFFFF], np.uint32)
    got = oracle.pcm_decode(pats.view(np.uint8), 1, pats.size, FLOAT)[0]
    assert np.array_equal(bits32(got), pats)
    # writing clamps to [-1, 1]: NaNs (payloads, signalling ones too), zeros and denormals keep their bits
    enc = oracle.pcm_encode(pats.view(np.float32)[None, :], FLOAT).view(np.uint32)
    x = pats.view(np.float32)
    want = np.where(np.isnan(x), pats, np.clip(x, -1, 1).view(np.uint32))
    assert np.array_equal(enc, want)
    assert enc[7] == 0x3F800000 and enc[8] == 0xBF800000 and enc[15] == 0x3F800000


def test_double_decode_rounds_to_nearest_even(oracle):
    tiny = 2.0 ** -149
    d = np.array([0.0, -0.0, 1.0, -1.0, 1 + 2.0 ** -24, 1 + 3 * 2.0 ** -24, 1 + 2.0 ** -24 + 2.0 ** -50, -(1 + 2.0 ** -24),
                  0.1, 1 / 3, 1e300, -1e300, 3.4028235677973366e38, 3.4028235e38, np.inf, -np.inf,
                  1e-50, -1e-50, tiny, tiny / 2, 3 * tiny / 2, tiny / 2 * 1.0000001, 2.0 ** -126 * (1 - 2.0 ** -25)], np.float64)
    got = oracle.pcm_decode(d.astype("<f8").view(np.uint8), 1, d.size, DOUBLE)[0]
    with np.errstate(over="ignore"):
        want = d.astype(F32)
    assert np.array_equal(bits32(got), bits32(want))
    assert got[4] == 1.0 and got[5] == F32(1 + 2.0 ** -22) and got[6] == F32(1 + 2.0 ** -23)
    assert np.isinf(got[10]) and np.isinf(got[12]) and got[13] == F32(3.4028235e38)
    assert got[16] == 0.0 and bits32(got)[17] == 0x80000000 and bits32(got)[18] == 1
    assert got[19] == 0.0 and bits32(got)[20] == 2 and bits32(got)[21] == 1
    assert bits32(got)[22] == 0x00800000                # rounds up out of the denormals


SCALE = {PCM_U8: 127.0, PCM_16: 32767.0, PCM_24: 8388607.0, PCM_32: 2147483648.0}


def expected_pcm(x, t):
    """The table's write rule in numpy: clamp, float32 product, round half to even; +1.0 and NaN special for PCM_32."""
    s = np.clip(x.astype(F32), F32(-1), F32(1))         # np.clip keeps NaN
    with np.errstate(invalid="ignore"):
        p = np.rint((s * F32(SCALE[t])).astype(F32)).astype(np.float64)
        q = np.where(np.isnan(s), -2.0 ** 31, p)
        if t == PCM_32:
            q = np.where(s == 1, -2.0 ** 31, q)
        q = q.astype(np.int64)
    if t == PCM_U8:
        q = q + 128
    return [(q >> (8 * k)) & 0xFF for k in range(WIDTH[t])]


def encode_ints(oracle, x, t):
    b = oracle.pcm_encode(x[None, :], t).reshape(-1, WIDTH[t]).astype(np.int64)
    return [b[:, k] for k in range(WIDTH[t])]


@pytest.mark.parametrize("t", [PCM_U8, PCM_16, PCM_24, PCM_32])
def test_pcm_encode_known_answers(oracle, t):
    special = np.array([1.0, -1.0, 0.0, -0.0, np.nan, np.inf, -np.inf, 1.5, -2.0, 1e30, 0.5, -0.5, 2.0 ** -32,
                        3 * 2.0 ** -32, 5 * 2.0 ** -32, np.float32(1 - 2.0 ** -24)], np.float32)
    # a grid of dyadic values: some of its products land exactly halfway between two integers (at least +-0.5)
    grid = (np.arange(-2 ** 14, 2 ** 14 + 1) / 2.0 ** 14).astype(np.float32)
    ties = (grid * F32(SCALE[t])).astype(F32)
    assert np.count_nonzero(ties - np.floor(ties) == 0.5) >= 2 or t == PCM_32
    rng = np.random.default_rng(t)
    x = np.concatenate([special, grid, rng.uniform(-1.2, 1.2, 5000).astype(np.float32)])
    got, want = encode_ints(oracle, x, t), expected_pcm(x, t)
    for k in range(WIDTH[t]):
        assert np.array_equal(got[k], want[k]), k
    v = sum(g << (8 * k) for k, g in enumerate(got))
    full = {PCM_U8: 255, PCM_16: 32767, PCM_24: 8388607, PCM_32: 0x80000000}[t]
    assert v[0] == full                                  # +1.0; PCM_32 wraps to INT_MIN as x86's lrintf gives it
    assert v[4] == (128 if t == PCM_U8 else (0x80000000 if t == PCM_32 else 0))     # NaN
    assert v[5] == v[0] and v[7] == v[0] and v[6] == v[1] and v[8] == v[1]          # clamped
    assert v[2] == v[3] == (128 if t == PCM_U8 else 0)


def test_pcm_encode_halfway_products_round_to_even(oracle):
    # 0.5 * 127 = 63.5 -> 64, 0.5 * 32767 = 16383.5 -> 16384, 0.5 * 8388607 = 4194303.5 -> 4194304,
    # 2^-32 * 2^31 = 0.5 -> 0, 3 * 2^-32 -> 1.5 -> 2, 5 * 2^-32 -> 2.5 -> 2
    x = np.array([[0.5, -0.5]], np.float32)
    assert list(oracle.pcm_encode(x, PCM_U8)) == [192, 64]
    assert list(oracle.pcm_encode(x, PCM_16).view("<i2")) == [16384, -16384]
    b = oracle.pcm_encode(x, PCM_24).reshape(2, 3).astype(np.int64)
    assert list(b[:, 0] | (b[:, 1] << 8) | (b[:, 2] << 16)) == [4194304, (1 << 24) - 4194304]
    y = np.array([[2.0 ** -32, 3 * 2.0 ** -32, 5 * 2.0 ** -32, -3 * 2.0 ** -32]], np.float32)
    assert list(oracle.pcm_encode(y, PCM_32).view("<i4")) == [0, 2, 2, -2]


def test_double_encode_is_exact(oracle):
    rng = np.random.default_rng(7)
    x = np.concatenate([np.array([1.0, -1.0, 0.0, -0.0, 2.0 ** -149, 1.5, -np.inf], np.float32),
                        rng.uniform(-1, 1, 1000).astype(np.float32)])
    got = oracle.pcm_encode(x[None, :], DOUBLE).view("<f8")
    assert np.array_equal(got.view(np.uint64), np.clip(x, -1, 1).astype(np.float64).view(np.uint64))
    assert np.isnan(oracle.pcm_encode(np.array([[np.nan]], np.float32), DOUBLE).view("<f8")[0])


def test_interleave_and_round_trip(oracle):
    rng = np.random.default_rng(3)
    x = rng.uniform(-1, 1, (3, 101)).astype(np.float32)
    for t in ALL:
        b = oracle.pcm_encode(x, t)
        assert b.size == 3 * 101 * WIDTH[t]
        # frame-major: the first frame's three channels come first
        for c in range(3):
            assert np.array_equal(b[c * WIDTH[t]:(c + 1) * WIDTH[t]], oracle.pcm_encode(x[c:c + 1, :1], t))
        y = oracle.pcm_decode(b, 3, 101, t)
        tol = {PCM_U8: 2 / 127, PCM_16: 2 / 32767, PCM_24: 2.0 ** -22, PCM_32: 2.0 ** -24, FLOAT: 0, DOUBLE: 0}[t]      # step + scale asymmetry
        assert np.max(np.abs(y - x)) <= tol


SCIPY_CASES = [(np.uint8, PCM_U8), (np.int16, PCM_16), (np.int32, PCM_32), (np.float32, FLOAT), (np.float64, DOUBLE)]


def scipy_values(dtype, n, C, seed):
    rng = np.random.default_rng(seed)
    if np.issubdtype(dtype, np.integer):
        info = np.iinfo(dtype)
        v = rng.integers(info.min, int(info.max) + 1, (n, C), dtype=np.int64).astype(dtype)
        v[0, 0], v[1, 0] = info.min, info.max
        return v
    v = rng.uniform(-1.5, 1.5, (n, C)).astype(dtype)
    v[0, 0] = -0.0
    return v


def expected_from_scipy(v, t):
    if t == PCM_U8:
        return (v.astype(np.int32) - 128).astype(F32) * F32(1 / 128)
    if t == PCM_16:
        return v.astype(F32) * F32(1 / 32768)
    if t == PCM_32:
        return v.astype(F32) * F32(2.0 ** -31)
    return v.astype(F32)


@pytest.mark.parametrize("dtype,t", SCIPY_CASES)
def test_scipy_files_decode_to_scipys_values(oracle, tmp_path, dtype, t):
    from scipy.io import wavfile
    C, n = 2, 1001
    v = scipy_values(dtype, n, C, t)
    path = str(tmp_path / "s.wav")
    wavfile.write(path, 44100, v)
    sr, back = wavfile.read(path)
    assert sr == 44100 and np.array_equal(back, v)
    got = oracle.pcm_decode(data_bytes(path), C, n, t)
    assert np.array_equal(bits32(got), bits32(expected_from_scipy(back, t).T))


def test_stdlib_wave_24_bit_file_decodes_to_its_values(oracle, tmp_path):
    C, n = 3, 777
    rng = np.random.default_rng(24)
    v = rng.integers(-2 ** 23, 2 ** 23, (n, C))
    v[0, :] = [-2 ** 23, 2 ** 23 - 1, 0]
    raw = np.stack([(v >> (8 * k)) & 0xFF for k in range(3)], -1).astype(np.uint8).tobytes()
    path = str(tmp_path / "w.wav")
    with wave.open(path, "wb") as w:
        w.setnchannels(C)
        w.setsampwidth(3)
        w.setframerate(48000)
        w.writeframes(raw)
    with wave.open(path, "rb") as w:
        frames = np.frombuffer(w.readframes(n), np.uint8).reshape(n, C, 3).astype(np.int64)
    ints = ((frames[..., 0] | (frames[..., 1] << 8) | (frames[..., 2] << 16)) << 40) >> 40      # sign-extend
    assert np.array_equal(ints, v)
    got = oracle.pcm_decode(data_bytes(path), C, n, PCM_24)
    assert np.array_equal(bits32(got), bits32((ints.astype(F32) * F32(2.0 ** -23)).T))
    # writing scales by 2^23 - 1, reading by 2^23 (libsndfile's asymmetry): the values come back within one code
    b = oracle.pcm_encode(got, PCM_24).reshape(n, C, 3).astype(np.int64)
    again = ((b[..., 0] | (b[..., 1] << 8) | (b[..., 2] << 16)) << 40) >> 40
    assert np.max(np.abs(again - v)) <= 1
