"""Every release instantiation of the analysis and resynthesis kernels, reached on the GPU at the shapes and edges that
select it, and checked against the oracle.

The launch policy (pv_policy.h: choose_analysis / choose_synthesis; tests/test_launch_policy.py checks it without a GPU)
picks the instantiation from the dft size, W == N, hop == N/16, whether the window fills whole slots, even hops, pointer
alignment, the resynthesis hint and the whole signal's frame count. Each test here names the instantiation its shape must
reach and reads the kernels the call launched from the CUDA profiler, so a change of policy cannot move a shape off the
path it is meant to test without a failure.

Each row asserts:
- the oracle gates of tests/parity.py (resynthesis gets the oracle's PV);
- a bound on the magnitude error of EVERY bin, quiet ones included:
      |m - m_ref| <= K * 2^-24 * log2(N) * rms_b(m_ref)      per frame.
  A float32 radix-r FFT of n points rounds each output through log_r(n) passes of butterflies whose twiddles carry a
  relative error of a few units of 2^-24; the error of an output is a sum of such roundings over all inputs, so by
  Parseval it scales with the frame's rms over bins, not with the bin's own level, and grows at most linearly in the
  number of passes. K = 16 covers the constant factors (complex multiply-add: up to 4 roundings per butterfly leg; the
  real-FFT unpack and the window product add one pass; hypotf one ulp) with room for the worst bin of a frame. The
  oracle's FFT runs in double and rounds once. The rms argument is weakest for tonal frames: there the loud bins' own
  roundings dominate and scale with the peak, up to sqrt(B) times the rms. The long sine sweeps of the hinted rows
  (dft 8192: 0.94 of the bound on a B200) come closest;
- power-of-two homogeneity, bit for bit: the input times 2^-8 gives m times 2^-8 and the same f, and PV magnitudes
  times 2^-12 give the output times 2^-12. This carries the checks at full level over to quiet signals, which the
  absolute resynthesis gate cannot see;
- bit-identical results where two instantiations or two paths serve the same shape.

The kernel names are read with torch.profiler (CUPTI records the library's launches on the same context as torch's).
If the profiler sees none of them, the module errors: the reach assertions are what this file is for."""
import re

import numpy as np
import pytest

from flan_b200.signals import noise_chirp, sine_sweep
from parity import assert_analysis_parity, assert_synthesis_parity

pytestmark = pytest.mark.gpu

SR = 48000.0
K_BOUND = 16.0
KERNEL = re.compile(r"\b(pv_\w+?_kernel)<([^<>]*)>")


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


def dev_offset(a, floats):
    """A contiguous CUDA copy of `a` that starts `floats` floats past an allocation's (512-byte aligned) start."""
    import torch
    a = np.ascontiguousarray(a, np.float32)
    buf = torch.empty(a.size + floats, dtype=torch.float32, device="cuda")
    view = buf[floats:].view(a.shape)
    view.copy_(torch.from_numpy(a))
    return view


def signal(C, n, seed):
    """C channels that cycle through noise + chirp, a full-band sine sweep and a quieter noise + chirp."""
    gens = [lambda: noise_chirp(n, SR, seed), lambda: sine_sweep(n, SR), lambda: noise_chirp(n, SR, seed + 1) * np.float32(0.25)]
    return np.stack([gens[c % 3]() for c in range(C)])


def kernel_names(events):
    """Normalised names ('pv_analysis_kernel<4096,16,512,true,false,false>') of this project's kernels."""
    out = set()
    for name in events:
        m = KERNEL.search(name)
        if m:
            out.add(m.group(1) + "<" + ",".join(s.strip() for s in m.group(2).split(",")) + ">")
    return out


def launched(fn):
    """(fn(), the set of this project's kernels the device ran during fn)."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, kernel_names(e.name for e in prof.events() if e.device_type == DeviceType.CUDA)


def min_blocks(threads, tps):
    return min(32, max(1, tps // threads))


def uses_tmem(name):
    """analysis_uses_tmem / synthesis_uses_tmem (pv_kernels.cu) for a normalised kernel name: 128 columns per CTA, at
    most 512 per SM, dft 4096 only (the analysis at 16 points per thread, the resynthesis in its standard-shape form)."""
    kind, args = name.split("<")
    args = args.rstrip(">").split(",")
    if kind == "pv_analysis_kernel":
        N, PT, TPS = (int(v) for v in args[:3])
        return N == 4096 and PT == 16 and min_blocks(N // (2 * PT), TPS) * 128 <= 512
    if kind == "pv_synthesis_mirror_kernel":
        N, TPS, GEN = int(args[0]), int(args[1]), args[3] == "true"
        return N == 4096 and not GEN and min_blocks(N // 32, TPS) * 128 <= 512
    return False


def reach_failures(names, stage, expect, tmem):
    """What is wrong with the kernels of one call: '' when `stage` ran exactly `expect`, whose tensor-memory use is `tmem`."""
    ran = {n for n in names if ("_" + stage + "_") in n}
    if ran != {expect}:
        return "%s reached %s, not %s" % (stage, sorted(ran), expect)
    if uses_tmem(expect) != tmem:
        return "%s: tensor memory %s, the table says %s" % (expect, uses_tmem(expect), tmem)
    return ""


def analysis_a(N):
    return "pv_analysis_kernel<%d,8,768,false,false,false>" % N


def analysis_b(N, pad=False, emit=False):
    return "pv_analysis_kernel<%d,16,512,true,%s,%s>" % (N, str(pad).lower(), str(emit).lower())


def synthesis_mirror(N, tps, one, gen):
    return "pv_synthesis_mirror_kernel<%d,%d,%s,%s>" % (N, tps, str(one).lower(), str(gen).lower())


def synthesis_plain(N, tps, one):
    return "pv_synthesis_kernel<%d,%d,%s>" % (N, tps, str(one).lower())


def all_bin_ratio(pv, pv_ref, N):
    """Largest |m - m_ref| / (K * 2^-24 * log2(N) * rms_b(m_ref)) over every bin of every frame. A frame whose reference
    is all zeros must be all zeros."""
    m = np.asarray(pv, np.float32)[..., 0].astype(np.float64)
    mr = np.asarray(pv_ref, np.float32)[..., 0].astype(np.float64)
    rms = np.sqrt(np.mean(mr * mr, axis=-1, keepdims=True))
    bound = K_BOUND * 2.0 ** -24 * np.log2(N) * rms
    err = np.abs(m - mr)
    assert not np.any((bound == 0) & (err != 0)), "a silent frame has non-zero magnitudes"
    return float(np.max(np.where(bound > 0, err / np.where(bound > 0, bound, 1.0), 0.0)))


def frame_windows(F):
    """Frames compared with the oracle: all of a short signal, else its head, middle and tail."""
    if F <= 160:
        return [(0, F)]
    return [(0, 48), (F // 2 - 40, F // 2 + 40), (F - 32, F)]


def check_analysis(eng, oracle, x, W, hop, N, place=dev, hint=False, label=""):
    """Runs the analysis of `x` (placed on the device by `place`), checks it against the oracle, the all-bin bound and
    power-of-two homogeneity, and returns (pv on the device, the kernels of the call)."""
    d = place(x)
    pv, names = launched(lambda: eng.convert_to_pv(d, SR, W, hop, N, for_resynthesis=hint))
    pv_np = pv.cpu().numpy()
    F = pv_np.shape[1]
    assert pv_np.shape == (x.shape[0], eng.num_frames(x.shape[1], hop), N // 2 + 1, 2)
    worst = 0.0
    for f0, f1 in frame_windows(F):
        ref = oracle.convert_to_pv(x, SR, W, hop, N, f0, f1)
        got = pv_np[:, f0:f1]
        assert_analysis_parity(got, ref, SR, hop, N, first_frame_has_history=f0 > 0)
        worst = max(worst, all_bin_ratio(got, ref, N))
    print("all-bin bound %s (W, hop, N) = (%d, %d, %d): largest ratio %.3g" % (label, W, hop, N, worst))
    assert worst <= 1.0, worst
    quiet = eng.convert_to_pv(place(x * np.float32(2.0 ** -8)), SR, W, hop, N, for_resynthesis=hint).cpu().numpy()
    assert np.array_equal(bits(quiet[..., 0]), bits(pv_np[..., 0] * np.float32(2.0 ** -8))), "m of the input * 2^-8"
    assert np.array_equal(bits(quiet[..., 1]), bits(pv_np[..., 1])), "f of the input * 2^-8"
    return pv, names


def check_synthesis(eng, oracle, W, hop, N, C=2, frames=240, seed=60):
    """Resynthesis of the oracle's PV of a C-channel signal: parity with the oracle and homogeneity. Returns (the PV on
    the host and the device, the output on the host, the kernels of the call)."""
    x = signal(C, (frames - 1) * hop, seed)
    pv = oracle.convert_to_pv(x, SR, W, hop, N)
    ar = oracle.analysis_rate(SR, hop)
    d = dev(pv)
    out, names = launched(lambda: eng.convert_to_audio(d, SR, float(ar), W))
    out = out.cpu().numpy()
    assert_synthesis_parity(out, oracle.convert_to_audio(pv, SR, ar, W))
    q = pv.copy()
    q[..., 0] *= np.float32(2.0 ** -12)
    quiet = eng.convert_to_audio(dev(q), SR, float(ar), W).cpu().numpy()
    assert np.array_equal(bits(quiet), bits(out * np.float32(2.0 ** -12))), "output of the magnitudes * 2^-12"
    return pv, d, out, names


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


@pytest.fixture(scope="module", autouse=True)
def profiler_sees_library(eng):
    """The profiler must see the library's kernels; without them no reach assertion of this file means anything. Which
    analysis kernel config 2's shape reaches is the rows' business: a policy change fails those, not every test."""
    x = dev(signal(2, 40 * 256, 1))
    _, names = launched(lambda: eng.convert_to_pv(x, SR, 4096, 256, 4096))
    if not any(n.startswith("pv_analysis_kernel<4096,") for n in names):
        raise RuntimeError("torch.profiler did not record the library's analysis kernel (it saw %s): this file cannot "
                           "tell which kernels its calls reach" % sorted(names))


# ---- analysis --------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("W,hop,N,C", [
    (256, 16, 256, 3),
    (300, 7, 512, 2),           # odd hop
    (1000, 100, 1024, 3),       # dft 1024 outside the mirrored shape
])
def test_analysis_8_points(eng, oracle, W, hop, N, C):
    x = signal(C, 300 * hop, 10)
    _, names = check_analysis(eng, oracle, x, W, hop, N)
    assert not reach_failures(names, "analysis", analysis_a(N), False), reach_failures(names, "analysis", analysis_a(N), False)


@pytest.mark.parametrize("side", ["below", "at"])
def test_analysis_2048_large_switch(eng, oracle, sms, side):
    """dft 2048 takes 16 points per thread from C * F >= sms * 128 whole-signal frames: one frame either side."""
    F = sms * 128 - (1 if side == "below" else 0)
    x = signal(1, (F - 1) * 128, 11)
    _, names = check_analysis(eng, oracle, x, 2048, 128, 2048, label=side)
    expect = analysis_a(2048) if side == "below" else analysis_b(2048)
    assert not reach_failures(names, "analysis", expect, False), reach_failures(names, "analysis", expect, False)


def test_analysis_mirror_1024(eng, oracle):
    x = signal(3, 300 * 64, 12)
    _, names = check_analysis(eng, oracle, x, 1024, 64, 1024)
    expect = "pv_analysis_mirror_kernel<1024,512>"
    assert not reach_failures(names, "analysis", expect, False), reach_failures(names, "analysis", expect, False)


@pytest.mark.parametrize("W,hop,N,C", [
    (4096, 256, 4096, 2),
    (3000, 100, 4096, 3),       # window not a whole number of slots
    (4096, 255, 4096, 2),       # odd hop: scalar loads
    (4096, 512, 4096, 3),       # W == N, hop != N/16
    (4096, 4096, 4096, 2),      # hop == W
    (64, 16, 4096, 3),          # a window of one partial slot
    (8192, 512, 8192, 2),
    (5000, 300, 8192, 3),
])
def test_analysis_16_points(eng, oracle, W, hop, N, C):
    x = signal(C, 200 * hop, 13)
    _, names = check_analysis(eng, oracle, x, W, hop, N)
    expect = analysis_b(N)
    assert not reach_failures(names, "analysis", expect, N == 4096), reach_failures(names, "analysis", expect, N == 4096)


@pytest.mark.parametrize("W,hop,N,C,large", [
    (2048, 128, 4096, 2, False),    # the API default shape
    (768, 96, 4096, 3, False),
    (256, 400, 4096, 2, False),     # one slot of window, hop > W
    (4096, 512, 8192, 2, False),
    (1024, 64, 2048, 2, True),      # dft 2048 takes 16 points per thread only above the frame threshold
])
def test_analysis_padded_window(eng, oracle, sms, W, hop, N, C, large):
    F = sms * 64 if large else 200
    x = signal(C, (F - 1) * hop, 14)
    _, names = check_analysis(eng, oracle, x, W, hop, N)
    expect = analysis_b(N, pad=True)
    assert not reach_failures(names, "analysis", expect, N == 4096), reach_failures(names, "analysis", expect, N == 4096)


def test_analysis_misaligned_input_leaves_the_padded_form(eng, oracle):
    """The API default shape with the input one float past an 8-byte boundary: aligned2 is false, the padded form's
    vector loads do not apply and the plain kernel runs. It gives the padded kernel's bits."""
    W, hop, N = 2048, 128, 4096
    x = signal(3, 200 * hop, 15)
    pv, names = check_analysis(eng, oracle, x, W, hop, N, place=lambda a: dev_offset(a, 1))
    expect = analysis_b(N)
    padded, names_padded = launched(lambda: eng.convert_to_pv(dev(x), SR, W, hop, N))
    assert np.array_equal(bits(pv.cpu().numpy()), bits(padded.cpu().numpy())), "plain kernel (offset input) != padded kernel"
    assert not reach_failures(names, "analysis", expect, True), reach_failures(names, "analysis", expect, True)
    padded_expect = analysis_b(N, pad=True)
    assert not reach_failures(names_padded, "analysis", padded_expect, True), reach_failures(names_padded, "analysis", padded_expect, True)


@pytest.mark.parametrize("W,hop,N", [
    (4096, 256, 4096),
    (4096, 128, 4096),
    (4096, 200, 4096),          # binc4 marks another set of bins for the scan to repair
    (8192, 512, 8192),
    (2048, 128, 2048),
])
def test_hinted_analysis_leaves_summaries(eng, oracle, sms, W, hop, N):
    """The hinted analysis (W == N) of two channels long enough for more than 256 resynthesis segments: the kernel that
    also leaves the phase summaries runs, its rows are the plain analysis's, and the promised resynthesis gives the plain
    one's samples and NaN flag bit for bit with one launch fewer. A shape whose hint is refused fails here."""
    import torch
    F = max(6000, sms * 64 + 1)         # past the dft-2048 frame threshold with two channels
    x = signal(2, (F - 1) * hop, 16)
    pv_h, names = check_analysis(eng, oracle, x, W, hop, N, hint=True)
    plain_pv, plain_names = launched(lambda: eng.convert_to_pv(dev(x), SR, W, hop, N))
    assert torch.equal(pv_h.view(torch.int32), plain_pv.view(torch.int32))
    # the same with digital silence and a NaN in the input: marked summaries, and a flag to agree on
    x[0, F * hop // 5:F * hop // 5 + 40 * hop] = 0.0
    x[1, F * hop // 2] = np.nan
    xd = dev(x)
    ar = eng.analysis_rate(SR, hop)
    counts = []
    for hinted in (True, False):
        pv = eng.convert_to_pv(xd, SR, W, hop, N, for_resynthesis=hinted)
        n0 = eng.launch_count()
        y, flag = eng.convert_to_audio(pv, SR, ar, W, check_nan=True, unchanged=hinted)
        counts.append(eng.launch_count() - n0)
        if hinted:
            y_h, flag_h = y, flag
    assert flag and flag_h
    assert torch.equal(y_h.view(torch.int32), y.view(torch.int32)), "promised resynthesis != plain resynthesis"
    expect = analysis_b(N, emit=True)
    failure = reach_failures(names, "analysis", expect, N == 4096)
    assert not failure, "the hint was refused or went elsewhere: " + failure
    plain_expect = analysis_b(N)
    assert not reach_failures(plain_names, "analysis", plain_expect, N == 4096), reach_failures(plain_names, "analysis", plain_expect, N == 4096)
    assert counts[0] == counts[1] - 1, "the promise saves exactly the phase summary launch: %s" % counts


# ---- resynthesis -----------------------------------------------------------------------------------------------------

def test_synthesis_4096_standard_shape_variants(eng, oracle):
    """The tensor-memory resynthesis at config 2's shape: the output does not depend on a PV that is only 8-byte
    aligned, on an output one float past an 8-byte boundary, or on cutting the output span to a few middle segments."""
    import torch
    W, hop, N = 4096, 256, 4096
    expect = synthesis_mirror(N, 512, True, False)
    pv, d, out, names = check_synthesis(eng, oracle, W, hop, N, C=3, frames=400)
    C, F = pv.shape[:2]
    ar = float(oracle.analysis_rate(SR, hop))
    failures = [reach_failures(names, "synthesis", expect, True)]
    d8 = dev_offset(pv, 2)
    assert d8.data_ptr() % 16 == 8
    y8, n8 = launched(lambda: eng.convert_to_audio(d8, SR, ar, W))
    assert np.array_equal(bits(y8.cpu().numpy()), bits(out)), "PV view 8-byte aligned"
    failures.append(reach_failures(n8, "synthesis", expect, True))
    buf = torch.empty(C * F * hop + 1, dtype=torch.float32, device="cuda")
    o1 = buf[1:].view(C, F * hop)
    _, n1 = launched(lambda: eng.convert_to_audio(d, SR, ar, W, out=o1))
    assert np.array_equal(bits(o1.cpu().numpy()), bits(out)), "output one float past an 8-byte boundary"
    failures.append(reach_failures(n1, "synthesis", expect, True))
    off, length = hop * (F // 2 - 24), hop * 48
    r, nr = launched(lambda: eng.convert_to_audio_range(d, 0, F, SR, ar, W, None, off, length))
    assert np.array_equal(bits(r.cpu().numpy()), bits(out[:, off:off + length])), "a middle span of the output"
    failures.append(reach_failures(nr, "synthesis", expect, True))
    assert not any(failures), failures


@pytest.mark.parametrize("W,hop,N,expect", [
    (1024, 64, 1024, synthesis_mirror(1024, 384, False, False)),
    (2048, 128, 2048, synthesis_mirror(2048, 384, False, False)),
    # general mirrored form: the window fills whole slots, even hop of at most one slot
    (2048, 128, 4096, synthesis_mirror(4096, 384, False, True)),
    (3072, 96, 4096, synthesis_mirror(4096, 384, False, True)),
    (4096, 128, 4096, synthesis_mirror(4096, 384, False, True)),
    (4096, 130, 4096, synthesis_mirror(4096, 384, False, True)),
    (256, 2, 4096, synthesis_mirror(4096, 384, False, True)),
    (1024, 64, 2048, synthesis_mirror(2048, 384, False, True)),
    (512, 32, 1024, synthesis_mirror(1024, 384, False, True)),
    (8192, 512, 8192, synthesis_mirror(8192, 512, True, False)),
    (4096, 256, 8192, synthesis_mirror(8192, 512, True, True)),
    # no mirrored form: hop above one slot, odd hops, windows of partial slots, small dfts
    (8192, 1024, 8192, synthesis_plain(8192, 1024, True)),
    (8192, 511, 8192, synthesis_plain(8192, 1024, True)),
    (4096, 255, 4096, synthesis_plain(4096, 768, False)),
    (4096, 512, 4096, synthesis_plain(4096, 768, False)),
    (3000, 100, 4096, synthesis_plain(4096, 768, False)),
    (256, 16, 256, synthesis_plain(256, 768, False)),
    (300, 7, 512, synthesis_plain(512, 768, False)),
    (1000, 50, 1024, synthesis_plain(1024, 768, False)),
    (2048, 127, 2048, synthesis_plain(2048, 768, False)),
])
def test_synthesis(eng, oracle, W, hop, N, expect):
    C = 3 if hop % 4 else 2
    _, _, _, names = check_synthesis(eng, oracle, W, hop, N, C=C)
    assert not reach_failures(names, "synthesis", expect, False), reach_failures(names, "synthesis", expect, False)
