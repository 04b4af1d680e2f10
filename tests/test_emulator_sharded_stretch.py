"""CPU test of the planned stretch run shard by shard (flan_b200_multi_stretch / _modify_time): each output shard reads
only the input rows of its window (stretch_window) from a buffer of its own and writes its segments into another, with
the row / segment offsets of StretchArgs. The result must equal the unsharded planned stretch bit for bit, for cuts at
pair boundaries, inside pairs, inside pairs that ended early (totalWeight == 0) and in the zero region below xpos[0].
Rows outside a window and cells outside a shard are NaN in the emulator, so a read or write past them shows."""
import ctypes

import numpy as np
import pytest


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


@pytest.fixture(scope="module")
def emu():
    from emu_lib import EmuModify
    e = EmuModify()
    i, f, i64 = ctypes.c_int, ctypes.c_float, ctypes.c_int64
    fp, i64p = ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_int64)
    e.L.pv_emu_stretch_sharded.restype = i64
    e.L.pv_emu_stretch_sharded.argtypes = [fp, i, i64, i, f, f, fp, fp, i64, i, i, i, i, ctypes.POINTER(i), fp, i64p, i, i64p]
    return e


def _fp(a):
    return None if a is None else a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))


def run(emu, pv, sr, ar, factor, seconds, seg_len, cuts_of):
    """(unsharded, sharded, row windows): cuts_of(out_frames) gives the inner cuts (multiples of seg_len)."""
    C, F, B, _ = pv.shape
    t, fs, bs = emu.view(factor if factor is not None else seconds, F, B)
    fa, se = (_fp(t), None) if factor is not None else (None, _fp(t))
    used = ctypes.c_int(0)
    frames = int(emu.L.pv_emu_stretch_sharded(_fp(pv), C, F, B, sr, ar, fa, se, fs, bs, 0, seg_len, 0, ctypes.byref(used),
                                              None, None, 0, None))
    assert frames > 0 and not used.value
    want = np.full((C, frames, B, 2), np.nan, np.float32)
    assert emu.L.pv_emu_stretch_sharded(_fp(pv), C, F, B, sr, ar, fa, se, fs, bs, 0, seg_len, 0, ctypes.byref(used),
                                        _fp(want), None, 0, None) == frames
    inner = sorted(set(int(c) for c in cuts_of(frames) if 0 < c < frames))
    assert all(c % seg_len == 0 for c in inner)
    cuts = np.array([0] + inner + [frames], np.int64)
    rows = np.zeros(2 * (len(cuts) - 1), np.int64)
    got = np.full_like(want, np.nan)
    i64p = ctypes.POINTER(ctypes.c_int64)
    assert emu.L.pv_emu_stretch_sharded(_fp(pv), C, F, B, sr, ar, fa, se, fs, bs, 0, seg_len, 0, ctypes.byref(used),
                                        _fp(got), cuts.ctypes.data_as(i64p), len(cuts) - 1, rows.ctypes.data_as(i64p)) == frames
    return want, got, rows.reshape(-1, 2), cuts


@pytest.fixture(scope="module")
def pv_case():
    rng = np.random.default_rng(11)
    C, F, B = 2, 90, 9
    pv = np.empty((C, F, B, 2), np.float32)
    pv[..., 0] = rng.uniform(0.0, 1.0, (C, F, B))
    pv[..., 1] = rng.uniform(-50.0, 20000.0, (C, F, B))
    pv[0, 20:24, 3, 0] = 0          # pairs of zero magnitudes: the pair ends at its first frame (PVModify.cpp:351-352)
    pv[1, 40:42, :, 0] = 0
    pv[0, 60, 5, 0] = 0             # one zero: the pair ends where the mix reaches it
    return pv, np.float32(48000.0), np.float32(48000.0 / 128)


EVERY = lambda frames: range(frames)                                          # noqa: E731 -- a cut at every frame
FEW = lambda frames: [frames // 7, frames // 3, frames // 3 + 1, frames - 2]    # noqa: E731


@pytest.mark.parametrize("factor", [2.0, 0.5, 3.3, "time-varying"])
def test_sharded_stretch_equals_unsharded(emu, pv_case, factor):
    pv, sr, ar = pv_case
    C, F, B, _ = pv.shape
    if factor == "time-varying":
        factor = np.random.default_rng(3).uniform(0.2, 4.0, (F, 1)).astype(np.float32)
    else:
        factor = np.float32(factor)
    for seg_len, cuts_of in [(1, EVERY), (1, FEW), (3, lambda n: [3 * (n // 9), 3 * (n // 6), 3 * (n // 3)]), (4, lambda n: [4])]:
        want, got, rows, cuts = run(emu, pv, sr, ar, factor, None, seg_len, cuts_of)
        assert np.array_equal(bits(got), bits(want)), (seg_len, cuts)
        for (r0, r1), x0, x1 in zip(rows, cuts[:-1], cuts[1:]):
            assert 0 <= r0 <= r1 <= F
            # a shard of one frame reads at most the pair around it (factor >= 0.2: a frame spans < 6 input frames)
            assert x1 - x0 > 1 or r1 - r0 <= 7


def test_sharded_modify_time_zero_head_and_flat_run(emu, pv_case):
    pv, sr, ar = pv_case
    C, F, B, _ = pv.shape
    t = np.arange(F, dtype=np.float32)[:, None] / ar
    m = t * np.float32(1.6) + np.float32(0.05)         # starts late: output frames below xpos[0] are zeros
    m[30:45] = m[30]                                   # a flat run: those pairs cover no output frame
    m = np.ascontiguousarray(m, np.float32)
    for seg_len, cuts_of in [(1, EVERY), (2, lambda n: [2, 10, 2 * (n // 4)])]:
        want, got, rows, cuts = run(emu, pv, sr, ar, None, m, seg_len, cuts_of)
        assert np.array_equal(bits(got), bits(want)), (seg_len, cuts)
        assert rows[0].tolist() == [0, 0]            # the first output frame lies in the zero head: no rows read
        assert not want[:, :2].any()
