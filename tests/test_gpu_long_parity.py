"""GPU parity at the lengths where the long-signal code paths run, against the oracle on the same seeded inputs.

Short signals never reach these paths, so the other parity tests cannot see them:
- the three-launch phase scan of resynthesis (more than 256 segments per channel) and its group-length doubling (more
  than 65 535 groups of 32 segments);
- the persistent repitch kernel with several rows per CTA (the row-ahead load and the two shared row buffers);
- the planned stretch, modify_time and the map check at config 4's frame count, and stretch_map's closed form for a
  constant at 2^24 frames and beyond;
- config 4's chain stage by stage;
- buffers with more than 2^31 floats and 2^31 MF elements.

Where the code claims exactness (the PV-domain chain, promised against plain resynthesis) the comparison is bit for
bit; elsewhere the gates of tests/parity.py apply. Each test also checks that it reached the path it is about."""
import ctypes

import numpy as np
import pytest

from flan_b200.signals import noise_chirp
from parity import assert_analysis_parity, assert_synthesis_parity

pytestmark = pytest.mark.gpu

SR = 48000.0


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


@pytest.fixture(scope="module")
def eng():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from flan_b200.engine import Engine
    return Engine(0)


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


def full(t, F, B):
    return np.ascontiguousarray(np.broadcast_to(np.asarray(t, np.float32).reshape(
        (F, 1) if np.shape(t) == (F, 1) else (1, -1) if np.ndim(t) == 1 else np.shape(t) or (1, 1)), (F, B)))


def launches(eng, fn):
    n0 = eng.launch_count()
    out = fn()
    return out, eng.launch_count() - n0


def assert_synthesis_parity_nan(audio, audio_ref, tol=1e-5):
    """assert_synthesis_parity where the signal carries a NaN: the same samples are NaN, the others meet the gate."""
    audio = np.asarray(audio, np.float32)
    audio_ref = np.asarray(audio_ref, np.float32)
    assert audio.shape == audio_ref.shape
    nan = np.isnan(audio_ref)
    assert nan.any() and np.array_equal(np.isnan(audio), nan)
    err = float(np.abs(audio[~nan].astype(np.float64) - audio_ref[~nan].astype(np.float64)).max())
    assert err <= tol, err
    return err


# ---- A. the three-launch phase scan --------------------------------------------------------------------------------

def scan_stress_channel(F, N, sr, hop, seed):
    """(m, f) rows that make the phase accumulator of resynthesis walk a hard path: frequency signs switch every 997
    frames (at every alignment to segments of at most 128 frames and groups of 32 of them) and the negative runs are a
    little faster, so the accumulator of those bins sinks below zero, where the reference stops wrapping it and the
    running maximum of the scan decides where it wraps again; bins at exactly 0 Hz; bins just inside +-sr/2."""
    B = N // 2 + 1
    rng = np.random.default_rng(seed)
    m = rng.uniform(0.02, 0.3, (F, B)).astype(np.float32)
    base = (np.arange(B) * (sr / N) + rng.uniform(-0.4, 0.4, B) * (sr / N)).astype(np.float64)
    sign = np.where((np.arange(F) // 997) % 2 == 0, 1.0, -1.06)
    f = sign[:, None] * base[None, :] + rng.uniform(-2.0, 2.0, (F, B))
    f[:, 0] = 0.0
    f[:, B // 3] = 0.0
    f[:, B - 1] = sr / 2 - 0.5
    f[:, B - 2] = -(sr / 2 - 0.25)
    f[:, B - 3] = sign * (sr / 2 - 1.0)
    return np.stack([m, f.astype(np.float32)], axis=-1)


def long_pv(oracle, W, hop, N, seconds, seed):
    """Two channels: the oracle's analysis of a noise + chirp signal and the synthetic stress channel."""
    n = int(SR * seconds)
    x = np.stack([noise_chirp(n, SR, seed)])
    analysed = oracle.convert_to_pv(x, SR, W, hop, N)[0]
    stress = scan_stress_channel(analysed.shape[0], N, SR, hop, seed + 1)
    return np.ascontiguousarray(np.stack([analysed, stress]))


@pytest.mark.parametrize("W,hop,N,seconds", [
    (1024, 64, 1024, 30.0),         # mirrored real-to-complex kernel
    (4096, 256, 4096, 180.0),       # config 2's kernel
    (2048, 128, 4096, 40.0),        # the API's default shape: general mirrored form
    (512, 32, 512, 20.0),           # 8-point kernel
    (96, 6, 96, 10.0),              # Bluestein (the oracle's DFT of this size is O(n^2): 1536 points cost 9 ms a frame)
])
def test_long_resynthesis_matches_oracle(eng, oracle, sms, W, hop, N, seconds):
    pv = long_pv(oracle, W, hop, N, seconds, 71)
    ar = oracle.analysis_rate(SR, hop)
    d_pv = dev(pv)
    F = pv.shape[1]
    if N == 96:     # 64-frame segments: more than the 8 persistent CTAs per SM the run-time-sized transform runs
        assert 2 * -(-F // 64) > 8 * sms
    out, n_long = launches(eng, lambda: eng.convert_to_audio(d_pv, SR, float(ar), W))
    # the same call at about 100 frames scans its segments in one launch: the long one takes two more
    _, n_short = launches(eng, lambda: eng.convert_to_audio(dev(pv[:, :100]), SR, float(ar), W))
    assert n_long == n_short + 2, (n_long, n_short)
    assert_synthesis_parity(out.cpu().numpy(), oracle.convert_to_audio(pv, SR, ar, W))


def test_hinted_long_resynthesis_repairs_marked_summaries(eng, oracle):
    """config 2's shape at 180 s through the hinted analysis: the analysis kernel leaves phase summaries with marked
    entries (the lowest bins, NaN / Inf), the three-launch scan repairs them, and the promised resynthesis gives the
    plain path's samples and NaN flag bit for bit. The input has stretches of digital silence and one NaN."""
    import torch
    W = N = 4096
    hop = 256
    n = int(SR * 180)
    x = np.stack([noise_chirp(n, SR, 81), noise_chirp(n, SR, 82) * np.float32(0.5)])
    for c, (a, b) in enumerate([(n // 7, n // 7 + 3 * 48000), (n // 2, n // 2 + 20 * W)]):
        x[c, a:b] = 0.0
    x[1, int(n * 0.9)] = np.nan
    xd = torch.from_numpy(x).cuda()
    ar = eng.analysis_rate(SR, hop)
    pv = eng.convert_to_pv(xd, SR, W, hop, N)
    plain, n_plain = launches(eng, lambda: eng.convert_to_audio(pv, SR, ar, W, check_nan=True))
    pv_h = eng.convert_to_pv(xd, SR, W, hop, N, for_resynthesis=True)
    assert torch.equal(pv_h.view(torch.int32), pv.view(torch.int32))
    hinted, n_hinted = launches(eng, lambda: eng.convert_to_audio(pv_h, SR, ar, W, check_nan=True, unchanged=True))
    assert n_hinted == n_plain - 1, "the promise saves exactly the phase summary launch"
    (y, flag), (y_h, flag_h) = plain, hinted
    assert flag and flag_h
    assert torch.equal(y_h.view(torch.int32), y.view(torch.int32))
    # the scan really is the three-launch one: the same call at about 100 frames launches two kernels fewer
    _, n_short = launches(eng, lambda: eng.convert_to_audio(pv[:, :100].contiguous(), SR, ar, W, check_nan=True))
    assert n_plain == n_short + 2
    pv_np = pv.cpu().numpy()
    assert_synthesis_parity_nan(y.cpu().numpy(), oracle.convert_to_audio(pv_np, SR, np.float32(ar), W))


def test_phase_scan_group_doubling_matches_oracle(eng, oracle):
    """More than 65 535 groups of 32 segments: the scan doubles its group length. (W, hop, N) = (4, 1, 4), mono: the
    segment length is at most 64 frames, so 64 * 32 * 65 536 frames and more need the doubling. (A window of 2 would
    do too, but its Hann window is zero at both ends and the output would be silence.)"""
    import torch
    W, hop, N = 4, 1, 4
    B = N // 2 + 1
    F = 64 * 32 * 65536 + 4099
    assert F > 64 * 32 * 65535
    g = torch.Generator(device="cuda").manual_seed(91)
    d_pv = torch.rand((1, F, B, 2), generator=g, device="cuda", dtype=torch.float32)
    d_pv[..., 1] = (d_pv[..., 1] - 0.48) * SR          # mostly positive, often negative, up to about +-sr/2
    ar = eng.analysis_rate(SR, hop)
    out, n_long = launches(eng, lambda: eng.convert_to_audio(d_pv, SR, ar, W))
    _, n_short = launches(eng, lambda: eng.convert_to_audio(d_pv[:, :100].contiguous(), SR, ar, W))
    assert n_long == n_short + 2
    out = out.cpu().numpy()
    pv = d_pv.cpu().numpy()
    del d_pv
    ref = oracle.convert_to_audio(pv, SR, np.float32(ar), W)
    assert np.abs(ref).max() > 0.1
    assert_synthesis_parity(out, ref)


# ---- B. the persistent repitch -------------------------------------------------------------------------------------

@pytest.mark.parametrize("N,T", [(2048, 256), (4096, 512), (8192, 1024), (16384, None)])
def test_persistent_repitch_matches_oracle(eng, oracle, sms, N, T):
    """At least 20 rows per CTA the persistent kernel can have resident (2048 / T per SM), so every CTA loads rows
    ahead and swaps its two shared row buffers many times. B = 8193 is past the shared kernel's 5120 bins: the general
    row kernel runs. Rows: an analysed channel and a channel of random frequencies."""
    import torch
    B = N // 2 + 1
    rows = 20 * sms * 2048 // (T or 1024)
    F = (rows + 1) // 2
    assert 2 * F >= 20 * sms * (2048 // (T or 1024))            # rows per possible CTA
    if T:
        assert B <= 5 * T and (T == 256 or B > 5 * (T // 2))    # the instantiation this B selects
    else:
        assert B > 5 * 1024                                      # past the shared kernel: the general row kernel
    hop = N // 4
    x = np.stack([noise_chirp((F - 1) * hop + 1, SR, 101)])
    pv_a = eng.convert_to_pv(dev(x), SR, N, hop, N)
    assert pv_a.shape[1] == F
    g = torch.Generator(device="cuda").manual_seed(102)
    pv_r = torch.rand((1, F, B, 2), generator=g, device="cuda", dtype=torch.float32)
    pv_r[..., 1] = (pv_r[..., 1] - 0.1) * (SR / 2)
    d_pv = torch.cat([pv_a, pv_r]).contiguous()
    del pv_a, pv_r
    pv = d_pv.cpu().numpy()
    rng = np.random.default_rng(103)
    tables = {
        "constant": np.float32(1.5),
        "ascending_row": rng.uniform(0.5, 2.0, B).astype(np.float32),
        "negative_row": rng.uniform(-2.0, -0.5, B).astype(np.float32),
        "mixed_sign_row": rng.uniform(-1.0, 2.0, B).astype(np.float32),     # plan refused: the row kernel runs
    }
    for interp in (0, 5, 9):
        for kind, t in tables.items():
            want = oracle.repitch(pv, SR, full(t, F, B), interp)
            got = eng.repitch(d_pv, SR, dev(t) if np.ndim(t) else float(t), interp).cpu().numpy()
            assert np.array_equal(bits(got), bits(want)), (kind, interp)
        Ff = 97
        t = rng.uniform(0.3, 2.5, (Ff, B)).astype(np.float32)               # full table: the row kernel, fewer rows
        sub = np.ascontiguousarray(pv[:, :Ff])
        want = oracle.repitch(sub, SR, t, interp)
        got = eng.repitch(dev(sub), SR, dev(t), interp).cpu().numpy()
        assert np.array_equal(bits(got), bits(want)), ("full", interp)


# ---- C. stretch and modify_time at config 4's length ---------------------------------------------------------------

C4_F, C4_B, C4_HOP = 675001, 33, 128       # config 4's 30 min at hop 128; dft 64


@pytest.fixture(scope="module")
def long_rows():
    rng = np.random.default_rng(111)
    pv = np.empty((1, C4_F, C4_B, 2), np.float32)
    pv[..., 0] = rng.uniform(0.0, 1.0, (1, C4_F, C4_B))
    pv[..., 1] = rng.uniform(-2000.0, SR / 2, (1, C4_F, C4_B))
    pv[0, 1000:1040, 3, 0] = 0.0                       # zero magnitudes: pairs that end early
    pv[0, 400000:400002, :, 0] = 0.0
    return pv


@pytest.mark.parametrize("kind", ["2.0", "0.5", "3.3", "1.0", "column", "per_bin"])
def test_long_stretch_bit_exact(eng, oracle, long_rows, kind):
    pv = long_rows
    F, B = C4_F, C4_B
    ar = oracle.analysis_rate(SR, C4_HOP)
    rng = np.random.default_rng(112)
    if kind == "column":        # time-varying: one factor per frame, shared by all bins (the planned kernel)
        ph = np.arange(F, dtype=np.float64) * (2 * np.pi / 90001)
        t = (1.2 + 0.7 * np.sin(ph) + rng.uniform(-0.05, 0.05, F)).astype(np.float32)[:, None]
    elif kind == "per_bin":     # a factor per (frame, bin): pv_stretch_kernel
        t = rng.uniform(0.5, 2.0, (F, B)).astype(np.float32)
    else:
        t = np.float32(float(kind))
    want = oracle.stretch(pv, SR, ar, full(t, F, B), 0)
    got = eng.stretch(dev(pv), SR, float(ar), dev(t) if np.ndim(t) else float(t), 0).cpu().numpy()
    assert got.shape == want.shape and np.array_equal(bits(got), bits(want)), kind


def test_long_modify_time_bit_exact(eng, oracle, long_rows):
    pv = long_rows
    F, B = C4_F, C4_B
    ar = oracle.analysis_rate(SR, C4_HOP)
    t = np.arange(F, dtype=np.float32) / np.float32(ar)
    late = t * np.float32(1.3) + np.float32(41.7)          # output starts 41.7 s in
    late[200000:260000] = late[200000]                     # a flat run
    to_3600 = t * np.float32(2.0) + np.float32(0.37)       # reaches about 3600 s: float positions 2.4e-4 s apart
    for name, m in [("late_start_flat_run", late), ("to_3600_s", to_3600)]:
        m = np.ascontiguousarray(m[:, None])
        want = oracle.modify_time(pv, SR, ar, full(m, F, B), 0)
        got = eng.modify_time(dev(pv), SR, float(ar), dev(m), 0).cpu().numpy()
        assert got.shape == want.shape and np.array_equal(bits(got), bits(want)), name
    assert want.shape[1] > 1349000


def test_long_stretch_summaries_and_resynthesis(eng, oracle, long_rows):
    """stretch(2.0) with summary_window: the promised resynthesis of its output is the plain one bit for bit and saves
    the phase summary launch; the plain one meets the gate against the oracle on the same rows."""
    import torch
    pv = long_rows
    W = 64
    ar = eng.analysis_rate(SR, C4_HOP)
    d_pv = dev(pv)
    st = eng.stretch(d_pv, SR, ar, 2.0, 0, summary_window=W)
    del d_pv
    promised, n_promised = launches(eng, lambda: eng.convert_to_audio(st, SR, ar, W, unchanged=True))
    plain, n_plain = launches(eng, lambda: eng.convert_to_audio(st, SR, ar, W))
    assert n_promised == n_plain - 1
    assert torch.equal(promised.view(torch.int32), plain.view(torch.int32))
    st_np = st.cpu().numpy()
    assert st_np.shape[1] == 2 * C4_F
    assert_synthesis_parity(plain.cpu().numpy(), oracle.convert_to_audio(st_np, SR, np.float32(ar), W))


def test_map_check_frame_count_matches_oracle(eng, oracle, sms):
    """The output frame count of modify_time comes from a grid-stride max over the map. Maps of more than twice the
    threads the check launches, so that every thread sees several elements, with the maximum in awkward places."""
    F, B = 20011, 33
    assert F * B > 2 * 8 * sms * 256                   # blocks are capped at 8 per SM, 256 threads each
    ar = eng.analysis_rate(SR, C4_HOP)
    rng = np.random.default_rng(121)
    base = rng.uniform(0.0, 900.0, (F, B)).astype(np.float32)
    maps = {}
    m = base.copy(); m[0, 0] = 1800.3; maps["max_first"] = m
    m = base.copy(); m[-1, -1] = 1800.3; maps["max_last"] = m
    m = base.copy(); m[5, 7] = m[F // 2, 3] = m[-3, 30] = 1234.5678; maps["max_repeated"] = m
    m = base.copy(); m[F - 1, 0] = 1000.0; m[1234, 5] = 999.9999; maps["max_last_row_first_bin"] = m
    maps["all_negative"] = -base - np.float32(0.01)
    m = -base - np.float32(0.01); m[F // 3, 11] = np.float32(-0.0); maps["max_negative_zero"] = m
    m = -base - np.float32(0.01); m[-1, -1] = np.float32(-0.0); m[0, 0] = np.float32(-0.0); maps["negative_zero_ends"] = m
    maps["ramp"] = np.ascontiguousarray(np.broadcast_to(np.arange(F, dtype=np.float32)[:, None] / np.float32(ar), (F, B)))
    for name, m in maps.items():
        m = np.ascontiguousarray(m, np.float32)
        frames = ctypes.c_int64(0)
        eng.ctx.call("flan_b200_modify_time_frames", eng._chk(dev(m)), B, 1, F, B, SR, ar, ctypes.byref(frames))
        want = oracle.L.pvo_modify_time(None, 1, F, B, SR, np.float32(ar), m.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), 0, None)
        assert frames.value == want, (name, frames.value, want)


@pytest.mark.parametrize("c", [1.0, 2.0, 0.7, 1.0 / 3.0])
def test_constant_stretch_map_at_2_24_frames(eng, c):
    """stretch_map of a constant factor uses a closed form per binade instead of F dependent float additions. Past 2^24
    frames the sum stops growing for c = 1 (and changes binade often for the others): the closed form must still give
    the sequential float32 running sum, divided by the rate, bit for bit."""
    F, B = (1 << 24) + 5000, 33
    ar = eng.analysis_rate(SR, C4_HOP)
    got = eng.stretch_map(F, B, SR, ar, float(c)).cpu().numpy()[:, 0]
    rate = np.float32(SR) / np.float32(C4_HOP)
    want = np.add.accumulate(np.full(F, c, np.float32), dtype=np.float32) / rate
    assert np.array_equal(bits(got), bits(want))


# ---- D. config 4's chain as bench.py --chain runs it ----------------------------------------------------------------

def test_config4_chain_stage_by_stage(eng, oracle):
    """One channel of config 4, 120 s: analysis -> repitch(1.5) -> stretch(2.0, summary_window) -> promised
    resynthesis, each stage fed the GPU's output of the stage before and compared with the oracle on that input."""
    import torch
    W = N = 2048
    hop = 128
    n = int(SR * 120)
    x = np.stack([noise_chirp(n, SR, 40)])
    ar32 = oracle.analysis_rate(SR, hop)
    ar = float(ar32)
    pv = eng.convert_to_pv(dev(x), SR, W, hop, N)
    pv_np = pv.cpu().numpy()
    assert_analysis_parity(pv_np, oracle.convert_to_pv(x, SR, W, hop, N), SR, hop, N)
    F, B = pv.shape[1], pv.shape[2]
    rp = eng.repitch(pv, SR, 1.5, 0)
    del pv
    rp_np = rp.cpu().numpy()
    assert np.array_equal(bits(rp_np), bits(oracle.repitch(pv_np, SR, np.full((F, B), 1.5, np.float32), 0)))
    del pv_np
    st = eng.stretch(rp, SR, ar, 2.0, 0, summary_window=W)
    st_np = st.cpu().numpy()
    assert np.array_equal(bits(st_np), bits(oracle.stretch(rp_np, SR, ar32, np.full((F, B), 2.0, np.float32), 0)))
    del rp
    promised, n_promised = launches(eng, lambda: eng.convert_to_audio(st, SR, ar, W, unchanged=True))
    plain, n_plain = launches(eng, lambda: eng.convert_to_audio(st, SR, ar, W))
    assert n_promised == n_plain - 1
    # the resynthesis of 2 F frames scans in three launches
    _, n_short = launches(eng, lambda: eng.convert_to_audio(st[:, :100].contiguous(), SR, ar, W))
    assert n_plain == n_short + 2
    assert torch.equal(promised.view(torch.int32), plain.view(torch.int32))
    assert_synthesis_parity(plain.cpu().numpy(), oracle.convert_to_audio(st_np, SR, ar32, W))


# ---- E. past 2^31 elements -----------------------------------------------------------------------------------------

def test_buffers_past_2_31_elements(eng, oracle):
    """100 channels of config 4's frame count at dft 64: C * F * B = 2.23e9 MF elements, past 2^31 MF elements and
    past 2^31 floats in one buffer. repitch(1.5), stretch(0.5) and a resynthesis at hop 16, each compared on channels
    either side of both boundaries with the oracle run on that channel alone. Peak device use is about 36 GB."""
    import torch
    C, F, B = 100, C4_F, C4_B
    N = W = 64
    hop = 16
    need = 2 * C * F * B * 8 + (1 << 32)
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip("needs %.1f GB of free device memory, %.1f GB free" % (need / 1e9, free / 1e9))
    per_channel = F * B
    assert 97 * per_channel > 1 << 31 > 96 * per_channel                 # MF elements: channel 96 holds 2^31
    assert 2 * 49 * per_channel > 1 << 31 > 2 * 48 * per_channel         # floats: channel 48 holds 2^31
    channels = [0, 48, 49, 96, 97, 99]
    ar32 = oracle.analysis_rate(SR, hop)
    ar = float(ar32)
    g = torch.Generator(device="cuda").manual_seed(131)
    torch.cuda.empty_cache()
    d_pv = torch.rand((C, F, B, 2), generator=g, device="cuda", dtype=torch.float32)
    d_pv[..., 1].sub_(0.05).mul_(SR / 2)           # in place: no second 18 GB temporary
    rows = {c: d_pv[c:c + 1].cpu().numpy() for c in channels}

    def const(v):
        return np.full((F, B), v, np.float32)

    out = eng.repitch(d_pv, SR, 1.5, 0)
    for c in channels:
        assert np.array_equal(bits(out[c:c + 1].cpu().numpy()), bits(oracle.repitch(rows[c], SR, const(1.5), 0))), c
    del out
    torch.cuda.empty_cache()

    out = eng.stretch(d_pv, SR, ar, 0.5, 0)
    assert out.shape[0] == C and C * out.shape[1] * B * 2 > 1 << 31
    for c in channels:
        want = oracle.stretch(rows[c], SR, ar32, const(0.5), 0)
        assert np.array_equal(bits(out[c:c + 1].cpu().numpy()), bits(want)), c
    del out
    torch.cuda.empty_cache()

    out = eng.convert_to_audio(d_pv, SR, ar, W)
    assert out.shape == (C, F * hop)
    for c in channels:
        assert_synthesis_parity(out[c:c + 1].cpu().numpy(), oracle.convert_to_audio(rows[c], SR, ar32, W))
    del out, d_pv
    torch.cuda.empty_cache()
