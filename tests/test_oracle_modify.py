"""CPU tests of the checker for the PV-domain chain (SURVEY 8f-1): the C restatement of PV::repitch / PV::stretch /
PV::modify_time (oracle/pv_oracle.c) against the reference's own PV/PVModify.cpp compiled verbatim
(oracle/_ref/libflan_ref_modify.so, or its results stored under tests/golden/reference/), bit for bit, and against the committed fixtures generated from that build."""
import glob
import os

import numpy as np
import pytest

from flan_b200.signals import make_config
from reference_records import Records, live_reference_modify

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "modify", "modify_*.npz")))


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


@pytest.fixture(scope="module")
def rec():
    r = Records("test_oracle_modify")
    yield r
    r.save()


@pytest.fixture(scope="module")
def pv_case(oracle):
    x, sr, W, h, N = make_config("cfg1", 0.25)
    return oracle.convert_to_pv(x, sr, W, h, N), sr, oracle.analysis_rate(sr, h), W


def tables(F, B):
    rng = np.random.default_rng(5)
    return {
        "const": np.full((F, B), 1.5, np.float32),
        "table": rng.uniform(0.5, 2.0, (F, B)).astype(np.float32),
        "signed": rng.uniform(-1.0, 2.0, (F, B)).astype(np.float32),
    }


@pytest.mark.parametrize("interp", range(10))
def test_modify_oracle_bit_identical_to_reference_build(oracle, rec, pv_case, interp):
    pv, sr, ar, W = pv_case
    _, F, B, _ = pv.shape
    ref = live_reference_modify()
    for kind, fac in tables(F, B).items():
        key = "interp%d.%s." % (interp, kind)
        rec.check(key + "repitch", oracle.repitch(pv, sr, fac, interp), None if ref is None else ref.repitch(pv, sr, ar, W, fac, interp))
        rec.check(key + "stretch", oracle.stretch(pv, sr, ar, fac, interp), None if ref is None else ref.stretch(pv, sr, ar, W, fac, interp))
        sec = np.cumsum(fac, axis=0, dtype=np.float32) / np.float32(ar)
        rec.check(key + "modify_time", oracle.modify_time(pv, sr, ar, sec, interp),
                  None if ref is None else ref.modify_time(pv, sr, ar, W, sec, interp))


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
def test_modify_oracle_reproduces_golden(oracle, path):
    g = np.load(path)
    sr, ar, interp = float(g["sr"]), float(g["analysis_rate"]), int(g["interp"])
    assert np.array_equal(bits(oracle.repitch(g["pv"], sr, g["repitch_factor"], interp)), bits(g["repitch"]))
    st = oracle.stretch(g["pv"], sr, ar, g["stretch_factor"], interp)
    assert st.shape == g["stretch"].shape and np.array_equal(bits(st), bits(g["stretch"]))


def test_modify_golden_fixtures_exist():
    assert len(GOLDEN) >= 3


def test_repitch_known_answers(oracle, pv_case):
    # factor 1: the running sum maps bin b to b + 1, pair (b-1, b) covers output bin b alone with mix 0, where
    # w0 < w1 is false and the pair's upper MF wins (PVModify.cpp:237): out.m[b] = m[b] for 1 <= b <= B-2; bin 0 is
    # never reached and the last pair's range is clamped away (PVModify.cpp:224-225).
    pv, sr, ar, W = pv_case
    _, F, B, _ = pv.shape
    out = oracle.repitch(pv, sr, np.ones((F, B), np.float32), 0)
    assert not out[:, :, B - 1].any() and not out[:, :, 0].any()
    m = pv[:, :, 1:B - 1, 0]
    assert np.array_equal(bits(out[:, :, 1:B - 1, 0]), bits(np.where(m > 0, m, np.float32(0))))


def test_stretch_known_answers(oracle, pv_case):
    # factor 1: the running sum maps frame k to k + 1 (up to the float rounding of frame_to_time / time_to_frame), so
    # pair (k-1, k) lands on output frame k with mix ~ 0: out[k] ~ pv[k-1]; output frame 0 is never reached.
    pv, sr, ar, W = pv_case
    _, F, B, _ = pv.shape
    out = oracle.stretch(pv, sr, ar, np.ones((F, B), np.float32), 0)
    assert abs(out.shape[1] - F) <= 1
    assert not out[:, 0].any()
    k = min(F, out.shape[1]) - 1
    assert np.allclose(out[:, 1:k, :, 0], pv[:, 0:k - 1, :, 0], rtol=1e-3, atol=1e-6)
    # factor 2 doubles the frame count
    assert abs(oracle.stretch(pv, sr, ar, np.full((F, B), 2.0, np.float32), 0).shape[1] - 2 * F) <= 1
