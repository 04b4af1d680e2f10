"""GPU parity tests of the PV-domain chain (SURVEY 8f-1): flan_b200_repitch / _modify_frequency / _stretch_map /
_modify_time through the C ABI against the oracle (PV/PVModify.cpp restated, pinned to the reference's own build):
bit-exact for interpolators 0-6 and 9, within an ulp for the two that go through cos / sin."""
import glob
import os

import numpy as np
import pytest

from flan_b200.signals import make_config

pytestmark = pytest.mark.gpu

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "modify", "modify_*.npz")))
EXACT_INTERPS = [0, 1, 2, 3, 4, 5, 6, 9]


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
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


@pytest.fixture(scope="module")
def pv_case(oracle):
    x, sr, W, h, N = make_config("cfg5", 0.2)
    pv = oracle.convert_to_pv(x, sr, W, h, N)
    pv = np.concatenate([pv, pv[:, ::-1] * np.float32(0.5)], axis=0)
    pv[0, 7, 100:140, 0] = 0
    pv[1, 30:34, :, 0] = 0
    return pv, sr, oracle.analysis_rate(sr, h)


def tables(F, B, lo, hi, seed):
    rng = np.random.default_rng(seed)
    return {
        "full": rng.uniform(lo, hi, (F, B)).astype(np.float32),
        "row": rng.uniform(lo, hi, (B,)).astype(np.float32),
        "column": rng.uniform(lo, hi, (F, 1)).astype(np.float32),
        "constant": np.float32(1.5),
    }


def full(t, F, B):
    t = np.asarray(t, np.float32)
    if t.ndim == 1:
        t = t[None, :]
    if t.ndim == 0:
        t = t.reshape(1, 1)
    return np.ascontiguousarray(np.broadcast_to(t, (F, B)))


def as_arg(t):
    return dev(t) if np.ndim(t) else float(t)


@pytest.mark.parametrize("interp", EXACT_INTERPS)
def test_repitch_bit_exact(eng, oracle, pv_case, interp):
    pv, sr, ar = pv_case
    _, F, B, _ = pv.shape
    d_pv = dev(pv)
    for lo, hi, seed in [(0.3, 2.5, 1), (-1.0, 2.0, 2), (-2.0, -0.1, 3)]:
        for kind, t in tables(F, B, lo, hi, seed).items():
            want = oracle.repitch(pv, sr, full(t, F, B), interp)
            got = eng.repitch(d_pv, sr, as_arg(t), interp).cpu().numpy()
            assert np.array_equal(bits(got), bits(want)), (kind, lo, hi)


@pytest.mark.parametrize("interp", EXACT_INTERPS)
def test_stretch_bit_exact(eng, oracle, pv_case, interp):
    pv, sr, ar = pv_case
    _, F, B, _ = pv.shape
    d_pv = dev(pv)
    for lo, hi, seed in [(0.0, 3.0, 4), (-1.0, 2.5, 5)]:
        for kind, t in tables(F, B, lo, hi, seed).items():
            want = oracle.stretch(pv, sr, ar, full(t, F, B), interp)
            got = eng.stretch(d_pv, sr, float(ar), as_arg(t), interp).cpu().numpy()
            assert got.shape == want.shape and np.array_equal(bits(got), bits(want)), (kind, lo, hi)


def test_modify_time_bit_exact(eng, oracle, pv_case):
    pv, sr, ar = pv_case
    _, F, B, _ = pv.shape
    rng = np.random.default_rng(6)
    t = np.arange(F, dtype=np.float32)[:, None] / np.float32(ar)
    maps = {
        "offset": (t * np.float32(1.7) + np.float32(0.05)) * np.ones((1, B), np.float32),
        "negative_start": (t * np.float32(0.9) - np.float32(0.02)) * np.ones((1, B), np.float32),
        "per_bin": t * rng.uniform(0.5, 2.0, (1, B)).astype(np.float32),
        "reversed": (t[::-1] * np.float32(1.3)) * np.ones((1, B), np.float32),
        "wobble": t + rng.uniform(-0.01, 0.01, (F, B)).astype(np.float32),
        "all_negative": -t - np.float32(1.0) + np.zeros((1, B), np.float32),
    }
    d_pv = dev(pv)
    for kind, m in maps.items():
        m = np.ascontiguousarray(m, np.float32)
        want = oracle.modify_time(pv, sr, ar, m, 0)
        got = eng.modify_time(d_pv, sr, float(ar), dev(m), 0).cpu().numpy()
        assert got.shape == want.shape and np.array_equal(bits(got), bits(want)), kind


def test_modify_frequency_bit_exact(eng, oracle, pv_case):
    pv, sr, ar = pv_case
    C, F, B, _ = pv.shape
    fac = np.random.default_rng(7).uniform(0.4, 2.0, (F, B)).astype(np.float32)
    hz = fac.copy()
    for b in range(1, B):
        hz[:, b] = fac[:, b] + hz[:, b - 1]
    dft = np.float32((B - 1) * 2)
    hz = hz * np.float32(sr) / dft
    bw = np.float32(sr) / dft
    fbin = np.clip(pv[..., 1] / bw, np.float32(0), np.float32(B - 1) - np.float32(0.0001)).astype(np.float32)
    lo = np.floor(fbin).astype(np.int64)
    r = fbin - lo.astype(np.float32)
    fr = np.arange(F)[None, :, None]
    in_mod = (hz[fr, lo] * (np.float32(1) - r) + hz[fr, lo + 1] * r).astype(np.float32)
    want = oracle.repitch(pv, sr, fac, 0)
    got = eng.modify_frequency(dev(pv), sr, dev(hz), dev(in_mod), 0).cpu().numpy()
    assert np.array_equal(bits(got), bits(want))


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p) for p in GOLDEN])
def test_modify_reproduces_golden(eng, path):
    g = np.load(path)
    sr, ar, interp = float(g["sr"]), float(g["analysis_rate"]), int(g["interp"])
    d_pv = dev(g["pv"])
    assert np.array_equal(bits(eng.repitch(d_pv, sr, dev(g["repitch_factor"]), interp).cpu().numpy()), bits(g["repitch"]))
    st = eng.stretch(d_pv, sr, ar, dev(g["stretch_factor"]), interp).cpu().numpy()
    assert st.shape == g["stretch"].shape and np.array_equal(bits(st), bits(g["stretch"]))


def test_sine_interpolators_within_an_ulp(eng, oracle, pv_case):
    pv, sr, ar = pv_case
    _, F, B, _ = pv.shape
    fac = np.full((F, B), 1.7, np.float32)
    for interp in (7, 8):
        want = oracle.stretch(pv, sr, ar, fac, interp)
        got = eng.stretch(dev(pv), sr, float(ar), 1.7, interp).cpu().numpy()
        assert got.shape == want.shape
        assert np.allclose(got, want, rtol=3e-6, atol=1e-9)
        assert np.mean(bits(got) == bits(want)) > 0.95


def test_wide_rows_and_many_frames(eng, oracle):
    # dft 8192 (4097 bins: 17 bins per thread of the row kernel) and a frame count that is not a multiple of the chunk
    x, sr, W, h, N = make_config("cfg3", 0.6)
    pv = oracle.convert_to_pv(x, sr, W, h, N)
    ar = oracle.analysis_rate(sr, h)
    _, F, B, _ = pv.shape
    d_pv = dev(pv)
    assert np.array_equal(bits(eng.repitch(d_pv, sr, 1.5, 0).cpu().numpy()), bits(oracle.repitch(pv, sr, np.full((F, B), 1.5, np.float32), 0)))
    want = oracle.stretch(pv, sr, ar, np.full((F, B), 2.0, np.float32), 0)
    got = eng.stretch(d_pv, sr, float(ar), 2.0, 0).cpu().numpy()
    assert got.shape == want.shape and np.array_equal(bits(got), bits(want))


def test_chain_properties_at_scale(eng):
    # cfg4-sized rows (1025 bins), 40 000 frames: size-independent properties. repitch( 1 ) keeps magnitudes of bins
    # 1..B-2 wherever they are positive; stretch by 2 doubles the frame count and every even output frame carries an
    # input frame's magnitudes (mix = 0 at the left frame of a pair).
    import torch
    F, B, sr, hop = 40000, 1025, 32768.0, 128        # analysis rate 256: frame <-> second conversions are exact
    ar = eng.analysis_rate(sr, hop)
    g = torch.Generator(device="cuda").manual_seed(11)
    pv = torch.rand((1, F, B, 2), generator=g, device="cuda", dtype=torch.float32)
    pv[..., 1] *= 16000.0
    rp = eng.repitch(pv, sr, 1.0, 0)
    assert torch.equal(rp[0, :, 1:B - 1, 0], pv[0, :, 1:B - 1, 0])
    assert not rp[0, :, 0].any() and not rp[0, :, B - 1].any()
    st = eng.stretch(pv, sr, ar, 2.0, 0)
    assert st.shape[1] == 2 * F
    assert torch.equal(st[0, 2:2 * F:2, :, 0], pv[0, 0:F - 1, :, 0])
    assert not st[0, :2].any()


@pytest.mark.parametrize("factor,frames", [(2.0, 3000), (0.7, 3000), (3.3, 300), (1.0, 40)])
def test_stretch_leaves_the_phase_summaries_resynthesis_needs(eng, factor, frames):
    """With summary_window set, the bin-shared stretch kernel also leaves the per-segment phase summaries of its output;
    convert_to_audio(unchanged=True) then skips pv_phase_seg_kernel (one launch fewer) and gives the same bits, the
    NaN / Inf pre-scan flag included. Summaries are dropped by anything that writes the rows or uses the scratch space."""
    import torch
    sr, W, hop, B = 48000.0, 2048, 128, 1025
    ar = eng.analysis_rate(sr, hop)
    g = torch.Generator(device="cuda").manual_seed(5)
    pv = torch.rand((2, frames, B, 2), generator=g, device="cuda", dtype=torch.float32)
    pv[..., 1] = (pv[..., 1] - 0.02) * 20000.0          # a few negative frequencies: the max-prefix part of the summaries
    pv[0, frames // 3, 5, 0] = 0.0
    pv[0, frames // 3 + 1, 5, 0] = 0.0                  # a pair of zero magnitudes: the pair ends early (PVModify.cpp:351-352)
    plain_st = eng.stretch(pv, sr, ar, factor, 0)
    plain, plain_flag = eng.convert_to_audio(plain_st, sr, ar, W, check_nan=True)
    st = eng.stretch(pv, sr, ar, factor, 0, summary_window=W)
    assert torch.equal(st, plain_st)
    n0 = eng.launch_count()
    reused, flag = eng.convert_to_audio(st, sr, ar, W, check_nan=True, unchanged=True)
    n_reused = eng.launch_count() - n0
    assert torch.equal(reused, plain) and flag == plain_flag and not flag
    n0 = eng.launch_count()
    eng.convert_to_audio(st, sr, ar, W)
    assert eng.launch_count() - n0 == n_reused + 1, "the reuse saves exactly the phase summary launch"
    # a NaN in the input reaches the output rows and the flag travels with the summaries
    bad = pv.clone()
    bad[1, frames // 2, 7, 1] = float("nan")
    st_bad = eng.stretch(bad, sr, ar, factor, 0, summary_window=W)
    _, flag_bad = eng.convert_to_audio(st_bad, sr, ar, W, check_nan=True, unchanged=True)
    _, flag_ref = eng.convert_to_audio(st_bad, sr, ar, W, check_nan=True)
    assert flag_bad == flag_ref
    # an unrelated call in between uses the scratch space: the promise finds nothing to reuse and the rows are read again
    st2 = eng.stretch(pv, sr, ar, factor, 0, summary_window=W)
    eng.convert_to_audio(plain_st, sr, ar, W)
    assert torch.equal(eng.convert_to_audio(st2, sr, ar, W, unchanged=True), plain)
    # a promise for rows that were overwritten since is the caller's lie; one for OTHER rows is simply ignored
    st3 = eng.stretch(pv, sr, ar, factor, 0, summary_window=W)
    assert torch.equal(eng.convert_to_audio(plain_st, sr, ar, W, unchanged=True), plain)
    del st3


def test_modify_time_per_bin_drops_the_summaries_of_the_rows_it_overwrites(eng):
    """The per-bin walk of modify_time writes rows without the scratch space. Summaries a stretch left for the same buffer
    must not survive it: a promise that the rows are unchanged since the last call that wrote them is then true, and
    resynthesis must read the new rows."""
    import ctypes
    import torch
    sr, W, hop, B, F = 48000.0, 2048, 128, 1025, 3000
    ar = eng.analysis_rate(sr, hop)
    g = torch.Generator(device="cuda").manual_seed(9)
    pv = torch.rand((2, F, B, 2), generator=g, device="cuda", dtype=torch.float32)
    pv[..., 1] *= 20000.0
    # a per-bin (B, 1) map that never descends and has the same maximum, hence the same output frame count (made first:
    # stretch_map uses the scratch space)
    seconds = eng.stretch_map(F, B, sr, ar, 2.0)
    scale = torch.linspace(0.9, 1.0, B, device="cuda")
    scale[-1] = 1.0
    per_bin = (seconds * scale[None, :]).contiguous()
    frames = ctypes.c_int64(0)
    eng.ctx.call("flan_b200_modify_time_frames", eng._chk(per_bin), B, 1, F, B, sr, ar, ctypes.byref(frames))
    Y = eng.stretch(pv, sr, ar, 2.0, 0, summary_window=W)
    before = Y.clone()
    assert frames.value == Y.shape[1]
    # the summaries are recorded: a promised resynthesis saves the phase summary launch (and publishes them again)
    n0 = eng.launch_count()
    eng.convert_to_audio(Y, sr, ar, W, unchanged=True)
    n_promised = eng.launch_count() - n0
    n0 = eng.launch_count()
    eng.convert_to_audio(Y, sr, ar, W)
    n_plain = eng.launch_count() - n0
    assert n_promised == n_plain - 1
    eng.ctx.call("flan_b200_modify_time", eng._chk(pv), 2, F, B, sr, ar, eng._chk(per_bin), B, 1, 0, frames.value,
                 eng._chk(Y), 0)
    assert not torch.equal(Y, before)
    n0 = eng.launch_count()
    after = eng.convert_to_audio(Y, sr, ar, W, unchanged=True)
    assert eng.launch_count() - n0 == n_plain, "the rows were overwritten: nothing to reuse"
    assert torch.equal(after, eng.convert_to_audio(Y, sr, ar, W))


def test_stretch_summaries_are_not_used_after_the_workspace_grows():
    """At a dft size of the run-time-sized transform (16384) resynthesis needs per-CTA slabs of scratch beside the phase
    summaries, more than the stretch asked for. On a fresh context the workspace then grows and loses what the stretch
    left: the promised resynthesis computes the summaries again (as many launches as the plain one) and gives the same
    bits. Once the workspace is large enough, the same promise saves the phase summary launch."""
    import torch
    from flan_b200.engine import Engine
    e = Engine(0)           # a context of its own: its workspace is sized by the calls below only
    sr, W, hop, B, F = 48000.0, 16384, 1024, 8193, 400
    ar = e.analysis_rate(sr, hop)
    g = torch.Generator(device="cuda").manual_seed(13)
    pv = torch.rand((1, F, B, 2), generator=g, device="cuda", dtype=torch.float32)
    pv[..., 1] *= 20000.0
    st = e.stretch(pv, sr, ar, 2.0, 0, summary_window=W)
    n0 = e.launch_count()
    promised = e.convert_to_audio(st, sr, ar, W, unchanged=True)
    n_promised = e.launch_count() - n0
    n0 = e.launch_count()
    plain = e.convert_to_audio(st, sr, ar, W)
    assert e.launch_count() - n0 == n_promised, "the workspace grew: the summaries must be computed again"
    assert torch.equal(promised, plain)
    st2 = e.stretch(pv, sr, ar, 2.0, 0, summary_window=W)
    n0 = e.launch_count()
    assert torch.equal(e.convert_to_audio(st2, sr, ar, W, unchanged=True), plain)
    assert e.launch_count() - n0 == n_promised - 1, "the workspace kept the summaries: one launch fewer"
