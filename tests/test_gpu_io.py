"""GPU parity tests of the file-format codecs (SURVEY 8f-4) through the C ABI: byte-exact against the oracle
(.flan codec pinned to the reference's own PVBuffer::save / load; PCM-24 restated from libsndfile) and against a file
written by the reference build itself."""
import ctypes
import os

import numpy as np
import pytest

from flan_b200.signals import noise_chirp
from reference_records import Records, file_codec_reference
from test_oracle_io import pv_fixture

pytestmark = pytest.mark.gpu


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


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


@pytest.mark.parametrize("shape", [(2, 9, 65), (1, 7, 129), (1, 1, 3), (3, 41, 1025)])
def test_flan_codec_byte_exact(eng, oracle, shape):
    C, F, B = shape
    pv, sr = pv_fixture(seed=F, C=C, F=F, B=max(B, 9) if B > 8 else 9)
    pv = np.ascontiguousarray(pv[:, :, :B])
    want = oracle.flan_encode(pv, sr)
    got = eng.flan_encode(dev(pv), sr).cpu().numpy()
    assert np.array_equal(got, want)
    back = eng.flan_decode(dev(want), (C, F, B), sr).cpu().numpy()
    assert np.array_equal(bits(back), bits(oracle.flan_decode(want, (C, F, B), sr)))


def test_flan_nan_and_inf_follow_the_reference_conversion(eng, oracle):
    pv = np.zeros((1, 1, 5, 2), np.float32)
    pv[0, 0, :, 0] = [np.nan, np.inf, -np.inf, 1.0, -1.0]
    pv[0, 0, :, 1] = [np.inf, np.nan, 3.0, -np.inf, 0.0]
    assert np.array_equal(eng.flan_encode(dev(pv), 48000.0).cpu().numpy(), oracle.flan_encode(pv, 48000.0))


@pytest.mark.parametrize("C,n", [(1, 1000), (2, 4099), (3, 12345), (8, 513)])
def test_pcm24_codec_byte_exact(eng, oracle, C, n):
    rng = np.random.default_rng(n)
    x = rng.uniform(-1.1, 1.1, (C, n)).astype(np.float32)
    x[0, :6] = [0.0, 1.0, -1.0, 0.5, 2.0 ** -24, -2.0 ** -23]
    want = oracle.pcm24_encode(x)
    assert np.array_equal(eng.pcm24_encode(dev(x)).cpu().numpy(), want)
    back = eng.pcm24_decode(dev(want), C, n).cpu().numpy()
    assert np.array_equal(bits(back), bits(oracle.pcm24_decode(want, C, n)))


@pytest.fixture(scope="module")
def rec():
    r = Records("test_gpu_io")
    yield r
    r.save()


def test_flan_files_interchange_with_the_reference_build(eng, oracle, rec, tmp_path):
    pv, sr = pv_fixture(seed=11, C=2, F=33, B=257)
    ar, W = oracle.analysis_rate(sr, 64), 512
    ours, theirs = str(tmp_path / "ours.flan"), str(tmp_path / "ref.flan")
    eng.save_flan(ours, dev(pv), sr, float(ar), W)
    ref = file_codec_reference()
    if ref is not None:
        ref.save_flan(theirs, pv, sr, ar, W)
    else:           # the file is ours, checked against the stored digest of the reference's, byte for byte
        theirs = ours
    # the same file, byte for byte
    rec.check("save.file", np.fromfile(ours, np.uint8), None if ref is None else np.fromfile(theirs, np.uint8))
    got, sr2, rate2, W2 = eng.load_flan(theirs)
    want, header = None, None
    if ref is not None:
        want, sr3, rate3, W3 = ref.load_flan(theirs)
        header = np.array([sr3, rate3, W3], np.float64)
    rec.check("load.header", np.array([sr2, rate2, W2], np.float64), header)
    rec.check("load.pv", got.cpu().numpy(), want)


def test_wav_files_round_trip_and_stdlib_reads_them(eng, oracle, tmp_path):
    import wave
    sr = 48000.0
    x = np.stack([noise_chirp(30001, sr, 1), noise_chirp(30001, sr, 2) * np.float32(3.0)])     # second channel clips
    path = str(tmp_path / "x.wav")
    eng.save_wav(path, dev(x), sr)
    with wave.open(path, "rb") as w:
        assert (w.getnchannels(), w.getsampwidth(), w.getframerate(), w.getnframes()) == (2, 3, 48000, 30001)
        assert w.readframes(30001) == oracle.pcm24_encode(x).tobytes()
    y, sr2 = eng.load_wav(path)
    assert sr2 == sr
    assert np.array_equal(bits(y.cpu().numpy()), bits(oracle.pcm24_decode(oracle.pcm24_encode(x), 2, 30001)))
    assert np.max(np.abs(y.cpu().numpy()[0] - x[0])) <= 2.0 ** -23


def test_cpp_api_files_either_side_of_the_path(oracle, tmp_path):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from flan_b200 import build
    build.build_host()
    L = ctypes.CDLL(build.api_test_path())
    fp, i, f = ctypes.POINTER(ctypes.c_float), ctypes.c_int, ctypes.c_float
    L.api_file_round_trip.argtypes = [fp, i, i, f, i, i, i, ctypes.c_char_p, ctypes.c_char_p, fp, fp, fp, fp]
    sr, W, h, N = 44100.0, 512, 64, 512
    n = 9000
    x = np.stack([noise_chirp(n, sr, 21), noise_chirp(n, sr, 22)])
    F, B = n // h + 1, N // 2 + 1
    la, lpv, rate, out = np.zeros_like(x), np.zeros((2, F, B, 2), np.float32), ctypes.c_float(), np.zeros((2, F * h), np.float32)
    p = lambda a: a.ctypes.data_as(fp)
    rc = L.api_file_round_trip(p(x), 2, n, sr, W, h, N, str(tmp_path / "a.wav").encode(), str(tmp_path / "a.flan").encode(),
                               p(la), p(lpv), ctypes.byref(rate), p(out))
    assert rc == F * h
    assert rate.value == h                                                  # the reference's load keeps the hop there
    assert np.array_equal(bits(la), bits(oracle.pcm24_decode(oracle.pcm24_encode(x), 2, n)))
    # the .flan file holds the engine's analysis of the loaded audio, quantised to 24 bits
    ref_pv = oracle.convert_to_pv(la, sr, W, h, N)
    q = oracle.flan_decode(oracle.flan_encode(ref_pv, sr), (2, F, B), sr)
    loud = ref_pv[..., 0] > 1e-2 * ref_pv[..., 0].max()
    assert np.max(np.abs(lpv[..., 0] - q[..., 0])[loud]) <= 1e-4 * ref_pv[..., 0].max()
    ref_out = oracle.convert_to_audio(lpv, sr, oracle.analysis_rate(sr, h), W)
    assert np.max(np.abs(out - ref_out)) <= 1e-5


def test_flan_decode_drops_the_summaries_of_the_rows_it_overwrites(eng):
    """flan_decode writes rows without the scratch space. Summaries an analysis left for the same buffer must not survive
    it: a promise that the rows are unchanged since the last call that wrote them is then true, and resynthesis must read
    the decoded rows."""
    import torch
    sr, N, hop = 48000.0, 4096, 256
    n = int(sr * 200)
    xd = torch.from_numpy(np.stack([noise_chirp(n, sr, 3), noise_chirp(n, sr, 5)])).cuda()
    ar = eng.analysis_rate(sr, hop)
    F, B = eng.num_frames(n, hop), N // 2 + 1
    other = eng.flan_encode(eng.convert_to_pv(xd.flip(1).contiguous(), sr, N, hop, N), sr)
    pv = torch.empty((2, F, B, 2), dtype=torch.float32, device="cuda")
    eng.convert_to_pv(xd, sr, N, hop, N, out=pv, for_resynthesis=True)
    # the summaries are recorded: a promised resynthesis saves the phase summary launch (and publishes them again)
    n0 = eng.launch_count()
    eng.convert_to_audio(pv, sr, ar, N, unchanged=True)
    n_promised = eng.launch_count() - n0
    n0 = eng.launch_count()
    eng.convert_to_audio(pv, sr, ar, N)
    n_plain = eng.launch_count() - n0
    assert n_promised == n_plain - 1
    eng._bind_stream()
    eng.ctx.call("flan_b200_flan_decode", eng._chk(other, torch.uint8), 2 * F * B, float(N), sr, eng._chk(pv))
    n0 = eng.launch_count()
    after = eng.convert_to_audio(pv, sr, ar, N, unchanged=True)
    assert eng.launch_count() - n0 == n_plain, "the rows were overwritten: nothing to reuse"
    assert torch.equal(after, eng.convert_to_audio(pv, sr, ar, N))
