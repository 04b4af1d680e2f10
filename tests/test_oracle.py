"""CPU tests of the checker itself: the C restatement (oracle/pv_oracle.c) against
 (1) the reference's own sources compiled verbatim (oracle/_ref), bit for bit, or where that build is absent its
     results as stored under tests/golden/reference/ (tests/reference_records.py);
 (2) the committed golden fixtures generated from that build (tests/golden/make_golden.py);
 (3) first-principles known answers that need no FFT library (SURVEY.md 8c pins 1-6).
"""
import glob
import os

import numpy as np
import pytest

from flan_b200.signals import make_config, noise_chirp
from reference_records import Records, live_reference

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz")))


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


@pytest.fixture(scope="module")
def rec():
    r = Records("test_oracle")
    yield r
    r.save()


def round_trip_matches_reference(oracle, ref, rec, key, x, sr, W, h, N, audio=True):
    """The checker's analysis, and its resynthesis of the reference's PV, equal the reference build's bit for bit."""
    pv_o = oracle.convert_to_pv(x, sr, W, h, N)
    ar = oracle.analysis_rate(sr, h)
    pv_r, ar_r = ref.convert_to_pv(x, sr, W, h, N) if ref is not None else (None, None)
    rec.check(key + ".analysis_rate", np.float32(ar), None if ref is None else np.float32(ar_r))
    rec.check(key + ".pv", pv_o, pv_r)
    if audio:       # pv_o equals the reference's PV here, so it stands in for it where the build is absent
        pv_in = pv_r if pv_r is not None else pv_o
        rec.check(key + ".audio", oracle.convert_to_audio(pv_in, sr, ar, W),
                  None if ref is None else ref.convert_to_audio(pv_in, sr, ar, W))


@pytest.mark.parametrize("name,sec", [("cfg1", 1.0), ("cfg2", 0.5), ("cfg3", 0.5), ("cfg5", 0.5)])
def test_oracle_bit_identical_to_reference_build(oracle, rec, name, sec):
    x, sr, W, h, N = make_config(name, sec)
    round_trip_matches_reference(oracle, live_reference(), rec, name, x, sr, W, h, N)


def test_oracle_bit_identical_zero_padded_and_odd_sizes(oracle, rec):
    x = np.stack([noise_chirp(5003, 32000, 9)])
    for W, h, N in [(256, 32, 1024), (512, 128, 512), (128, 8, 256), (1000, 100, 1024)]:
        round_trip_matches_reference(oracle, live_reference(), rec, "odd_%d_%d_%d" % (W, h, N), x, 32000, W, h, N)


def test_oracle_bit_identical_at_any_dft_size(oracle, rec):
    """FFTW plans any size (FFTHelper.cpp:16-26): the restatement follows the reference build's stand-in (radix-2 for
    powers of two, the O(n^2) definition in long double otherwise) at small, non-power-of-two and odd sizes. For an odd
    dft size the reference derives bin frequencies -- and, in convert_to_audio, the inverse transform's size -- from
    get_dft_size() = (num_bins - 1) * 2 (PVBuffer.cpp:356-359,443-446), i.e. from dft_size - 1."""
    x = np.stack([noise_chirp(2100, 32000, 11)])
    for W, h, N in [(64, 8, 64), (100, 10, 128), (300, 30, 300), (96, 12, 192), (250, 25, 375), (201, 20, 201), (120, 15, 255)]:
        # the inverse runs at (num_bins - 1) * 2 points: the window must still fit
        round_trip_matches_reference(oracle, live_reference(), rec, "dft_%d_%d_%d" % (W, h, N), x, 32000, W, h, N,
                                     audio=W <= (N // 2) * 2)


def test_oracle_hann_matches_reference_build(oracle, rec):
    ref = live_reference()
    for W in (64, 1000, 2048, 8192):
        rec.check("hann_%d" % W, oracle.hann(W), None if ref is None else ref.hann(W))


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
def test_oracle_reproduces_golden(oracle, path):
    g = np.load(path)
    sr, W, h, N = float(g["sr"]), int(g["W"]), int(g["hop"]), int(g["N"])
    pv = oracle.convert_to_pv(g["audio_in"], sr, W, h, N)
    assert np.array_equal(bits(pv), bits(g["pv"]))
    audio = oracle.convert_to_audio(g["pv"], sr, g["analysis_rate"], W)
    assert np.array_equal(bits(audio), bits(g["audio_out"]))
    assert np.array_equal(bits(oracle.hann(W)), bits(g["hann"]))
    if "pv_ms" in g:
        ms = oracle.mid_side(g["audio_in"])
        assert np.array_equal(bits(oracle.convert_to_pv(ms, sr, W, h, N)), bits(g["pv_ms"]))
        lr = oracle.mid_side(oracle.convert_to_audio(g["pv_ms"], sr, g["analysis_rate"], W))
        assert np.array_equal(bits(lr), bits(g["audio_lr"]))


def test_golden_fixtures_exist():
    assert len(GOLDEN) >= 4


# ---------- first-principles known answers (no FFT library involved) ----------

def test_frame_count_and_output_length(oracle):
    # F = floor(n/h) + 1 (AudioPV.cpp:17); output length F*h (AudioPV.cpp:93)
    assert oracle.num_frames(441000, 128) == 3446
    assert oracle.num_frames(28800000, 256) == 112501
    assert oracle.num_frames(127, 128) == 1
    x = np.zeros((1, 1000), np.float32)
    pv = oracle.convert_to_pv(x, 8000, 64, 16, 64)
    assert pv.shape == (1, 63, 33, 2)
    assert oracle.convert_to_audio(pv, 8000, oracle.analysis_rate(8000, 16), 64).shape == (1, 63 * 16)


def test_all_zero_input_known_answer(oracle):
    # arg(0) = 0 so phase_diff = 0 and f[b] = binf + wrap(-expected[b]) * ar / pi2, m = 0.
    sr, W, h, N = 48000.0, 256, 16, 256
    pv = oracle.convert_to_pv(np.zeros((1, 2000), np.float32), sr, W, h, N)
    assert np.all(pv[..., 0] == 0)
    pi2 = np.float32(np.float32(np.arccos(np.float32(-1.0))) * np.float32(2))
    ar = np.float32(sr) / np.float32(h)
    b = np.arange(N // 2 + 1, dtype=np.float32)
    binf = b * np.float32(sr) / np.float32(N)
    expected = binf / ar * pi2
    delta = np.float32(0) - expected
    q = delta / pi2
    r = np.where(q >= 0, np.floor(q + np.float32(0.5)), -np.floor(-q + np.float32(0.5))).astype(np.float32)
    wrapped = delta - pi2 * r
    f = binf + wrapped * ar / pi2
    assert np.array_equal(bits(pv[0, 5, :, 1]), bits(f.astype(np.float32)))
    # half-way case: expected = pi -> roundf(-0.5) = -1 -> f = binf + ar/2
    k = N // (2 * h)
    assert pv[0, 5, k, 1] == binf[k] + ar / 2


def test_unit_impulse_known_answer(oracle):
    # frame 0 is centred on sample 0: only hann[W/2] survives, |X[b]| = hann[W/2] for every bin.
    W = 128
    x = np.zeros((1, 1024), np.float32)
    x[0, 0] = 1.0
    pv = oracle.convert_to_pv(x, 8000, W, 16, W)
    hann = oracle.hann(W)
    assert np.allclose(pv[0, 0, :, 0], hann[W // 2], rtol=1e-6)


def test_bin_centred_sine_known_answer(oracle):
    sr, W, h = 48000.0, 1024, 64
    k0, A = 37, 0.5
    n = 20000
    t = np.arange(n, dtype=np.float64)
    x = (A * np.sin(2 * np.pi * k0 * t / W)).astype(np.float32)[None]
    pv = oracle.convert_to_pv(x, sr, W, h, W)
    interior = pv[0, 20:-20]
    assert np.all(np.argmax(interior[..., 0], axis=1) == k0)
    assert np.allclose(interior[:, k0, 0], A * W / 4, rtol=2e-3)
    assert np.allclose(interior[:, k0, 1], k0 * sr / W, atol=0.05)


def test_round_trip_gain_of_steady_sine(oracle):
    # sum_i hann^2 = 3W/8 and the 2.67f constant (AudioPV.cpp:99) give a gain of ~1.001
    sr, W, h = 44100.0, 1024, 64
    n = 30000
    x = (0.5 * np.sin(2 * np.pi * 1000.0 * np.arange(n) / sr)).astype(np.float32)[None]
    pv = oracle.convert_to_pv(x, sr, W, h, W)
    y = oracle.convert_to_audio(pv, sr, oracle.analysis_rate(sr, h), W)
    g = np.sqrt(np.mean(y[0, 4096:n - 4096] ** 2) / np.mean(x[0, 4096:n - 4096] ** 2))
    assert 0.999 < g < 1.003


def test_ms_wrappers_null_unless_stereo(rec):
    """convert_to_ms_PV returns a null PV unless the audio is stereo (AudioPV.cpp:82): the reference build does, and so
    does this project's C++ API, which follows it (frames returned, -1 for a null PV)."""
    import ctypes
    from flan_b200 import build
    build.build_host()
    api = ctypes.CDLL(build.api_test_path())
    fp = ctypes.POINTER(ctypes.c_float)
    api.api_convert_to_pv.argtypes = [fp, ctypes.c_int, ctypes.c_int, ctypes.c_float, ctypes.c_int, ctypes.c_int,
                                      ctypes.c_int, ctypes.c_int, fp, fp]
    ref = live_reference()
    for C in (1, 3):
        x = np.zeros((C, 4096), np.float32)
        pv, ar = np.zeros((C, 129, 129, 2), np.float32), np.zeros(1, np.float32)
        frames = api.api_convert_to_pv(x.ctypes.data_as(fp), C, 4096, 48000.0, 256, 32, 256, 1, pv.ctypes.data_as(fp),
                                       ar.ctypes.data_as(fp))
        theirs = None
        if ref is not None:
            pv_r, _ = ref.convert_to_pv(x, 48000, 256, 32, 256, ms=True)
            theirs = np.array([-1 if pv_r is None else pv_r.shape[1]], np.int64)
        rec.check("ms_pv_frames_%dch" % C, np.array([frames], np.int64), theirs)


def test_chunked_oracle_equals_full(oracle):
    x, sr, W, h, N = make_config("cfg5", 0.5)
    full = oracle.convert_to_pv(x, sr, W, h, N)
    part = oracle.convert_to_pv(x, sr, W, h, N, 100, 231)
    assert np.array_equal(bits(full[:, 100:231]), bits(part))
