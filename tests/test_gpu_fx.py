"""Expression Functions on the GPU: the grid sampler and the at-PV evaluator (flan_b200_fx_sample / _fx_at_pv) against
the host evaluator they share their source with; PV::repitch / stretch / modify_time / modify_frequency with an
expression against the same call with its lambda, bit for bit (tests/cpp/fx_driver.cpp); the kernels each route reaches;
and a time-only stretch that keeps a PV sharded over several devices."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from flan_b200 import capi
from flan_b200.signals import noise_chirp, sine_sweep

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.fixture(scope="module")
def eng():
    from flan_b200.engine import Engine
    return Engine(0)


@pytest.fixture(scope="module")
def drv():
    from flan_b200 import build
    build.build_host()
    L = ctypes.CDLL(build.fx_test_path())
    i, fp, ip = ctypes.c_int, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_int)
    L.fx_chain.argtypes = [fp, i, i, ctypes.c_float, i, i, i, i, i, i, i, fp, ip, fp, ip]
    L.fx_refusals.argtypes = [fp, i, ctypes.c_float]
    return L


def host_eval(lib, prog, t, f):
    out = ctypes.c_float()
    assert lib.flan_b200_fx_eval(ctypes.byref(prog), float(t), float(f), ctypes.byref(out)) == 0
    return out.value


EXACT = capi.fx_program(["t", 0.5, "mul", "f", 1000.0, "div", "add", "t", "floor", "f", "sqrt", "max", "sub",
                         "t", 3.0, "lt", ("curve", 0), "f", 9000.0, "gt", "where"],
                        [([(0.0, 1.0), (1.0, 1.5), (2.0, 0.25)], 5)])
TRANSCENDENTAL = capi.fx_program(["t", 7.0, "mul", "sin", "f", 1.0, "add", "log", "mul", "t", -0.25, "mul", "exp", "add",
                                  "f", 0.001, "mul", "cos", 1.5, "pow", "add"])
T_ONLY = capi.fx_program(["t", ("curve", 0), 0.5, "mul"], [([(0.0, 1.0), (10.0, 2.0), (20.0, 0.5)], 6)])
F_ONLY = capi.fx_program(["f", 24000.0, "div", 1.0, "add"])
NEITHER = capi.fx_program([1.25, 0.25, "add"])


def grid(lib, prog, F, B, ts, bw, rows=None):
    """Host evaluation of rows (all when None) of the grid: value( x, y ) = program( float( x ) * ts, float( y ) * bw )."""
    xs = np.arange(F, dtype=np.float32) if rows is None else np.array(rows, np.float32)
    tx, fy = (xs * f32(ts)).tolist(), (np.arange(B, dtype=np.float32) * f32(bw)).tolist()
    out, fn, p = ctypes.c_float(), lib.flan_b200_fx_eval, ctypes.byref(prog)
    res = np.empty((len(tx), B), np.float32)
    for i, t in enumerate(tx):
        for j, f in enumerate(fy):
            fn(p, t, f, ctypes.byref(out))
            res[i, j] = out.value
    return res


def compare(got, want, exact, label):
    """Bit for bit (NaN included: both sides return the one quiet NaN 0x7fc00000), or within one ulp for programs with
    transcendental ops."""
    if exact:
        assert np.array_equal(bits(got), bits(want)), label
        return 0
    d = np.abs(bits(got).astype(np.int64) - bits(want).astype(np.int64))
    assert d.max() <= 1, (label, int(d.max()))
    n = int((d > 0).sum())
    print("%s: %d of %d values differ by one ulp" % (label, n, d.size))
    return n


@pytest.mark.parametrize("shape", ["cfg1", "odd"])
@pytest.mark.parametrize("name", ["exact", "transcendental", "t_only", "f_only", "neither"])
def test_sampler_equals_host_evaluator(eng, shape, name):
    prog = {"exact": EXACT, "transcendental": TRANSCENDENTAL, "t_only": T_ONLY, "f_only": F_ONLY, "neither": NEITHER}[name]
    sr, hop, N = (44100.0, 128, 2048) if shape == "cfg1" else (22050.0, 37, 250)
    F, B = (441000 // hop + 1, N // 2 + 1) if shape == "cfg1" else (301, 126)
    ts, bw = f32(1.0) / f32(eng.analysis_rate(sr, hop)), f32(sr) / f32(N)
    got = eng.fx_sample(prog, F, B, ts, bw).cpu().numpy()
    rows = F if prog is not F_ONLY and prog is not NEITHER else 1
    cols = B if prog is not T_ONLY and prog is not NEITHER else 1
    assert got.size == rows * cols
    want = grid(eng.lib, prog, rows, cols, ts, bw)
    compare(got.reshape(rows, cols), want, prog is not TRANSCENDENTAL, "%s %s" % (name, shape))


@pytest.mark.parametrize("name", ["exact", "transcendental"])
def test_sampler_on_a_config4_channel_grid(eng, name):
    # one config-4 channel: 30 min at 48 kHz, hop 128, dft 2048 -> 675001 x 1025 values (2.77 GB); seeded rows checked
    prog = EXACT if name == "exact" else TRANSCENDENTAL
    sr, hop, N = 48000.0, 128, 2048
    F, B = 48000 * 1800 // hop + 1, N // 2 + 1
    ts, bw = f32(1.0) / f32(eng.analysis_rate(sr, hop)), f32(sr) / f32(N)
    got = eng.fx_sample(prog, F, B, ts, bw)
    rows = sorted({0, 1, F - 1, F // 2} | set(np.random.default_rng(5).integers(0, F, 12).tolist()))
    sel = got[rows].cpu().numpy()
    del got
    compare(sel, grid(eng.lib, prog, F, B, ts, bw, rows), name == "exact", "cfg4 " + name)


@pytest.mark.parametrize("name", ["exact", "transcendental"])
def test_at_pv_equals_host_evaluator(eng, name):
    import torch
    prog = EXACT if name == "exact" else TRANSCENDENTAL
    C, F, B = 2, 203, 129
    rng = np.random.default_rng(9)
    pv = np.stack([rng.uniform(0, 1, (C, F, B)), rng.uniform(-100, 24000, (C, F, B))], axis=-1).astype(np.float32)
    pv[0, 3, :8, 1] = [0.0, -0.0, np.inf, -np.inf, np.nan, 1e-40, 3e38, 16777217.0]
    sr, hop = 48000.0, 128
    frame_rate = f32(sr) / f32(hop)
    got = eng.fx_at_pv(prog, torch.from_numpy(pv).cuda(), frame_rate).cpu().numpy()
    want = np.array([[[host_eval(eng.lib, prog, f32(x) / frame_rate, pv[c, x, b, 1]) for b in range(B)] for x in range(F)]
                     for c in range(C)], np.float32)
    compare(got, want, name == "exact", "at_pv " + name)


SR, W, HOP, N = 48000.0, 512, 64, 512


def signal(n=12000, C=2):
    return np.stack([noise_chirp(n, SR, 8), sine_sweep(n, SR)][:C]).astype(np.float32)


def chain(drv, x, op, cls, interp, lam):
    """(pv, audio, input host vector current) of the driver's fx_chain."""
    C, n = x.shape
    F, B = n // HOP + 1, N // 2 + 1
    cap = 4 * F + 64
    pv = np.zeros((C, cap, B, 2), np.float32)
    y = np.zeros((C, cap * HOP), np.float32)
    frames, host = ctypes.c_int(0), ctypes.c_int(-1)
    fp = ctypes.POINTER(ctypes.c_float)
    got = drv.fx_chain(x.ctypes.data_as(fp), C, n, SR, W, HOP, N, op, cls, interp, lam, pv.ctypes.data_as(fp),
                       ctypes.byref(frames), y.ctypes.data_as(fp), ctypes.byref(host))
    assert got == frames.value * HOP, (op, cls, interp, lam, got)
    # fx_chain copies C * frames * B MF contiguously: re-view the start of the buffer as [C, frames, B]
    flat = pv.reshape(-1)[:C * frames.value * B * 2].reshape(C, frames.value, B, 2)
    return flat, y.reshape(-1)[:C * got].reshape(C, got), host.value


@pytest.mark.parametrize("interp", [0, 2, 5, 9])
@pytest.mark.parametrize("op", [0, 1, 2, 3], ids=["repitch", "stretch", "modify_time", "modify_frequency"])
def test_expression_equals_its_lambda(drv, op, interp):
    x = signal()
    for cls in range(5):
        pe, ye, _ = chain(drv, x, op, cls, interp, 0)
        pl, yl, _ = chain(drv, x, op, cls, interp, 1)
        assert pe.shape == pl.shape and np.array_equal(bits(pe), bits(pl)), (op, cls, interp)
        assert np.array_equal(bits(ye), bits(yl)), (op, cls, interp)
        # a time map flat in time, or a frequency map that sends every bin of a frame to one frequency (it does not
        # read f), leaves nothing audible
        if not (op == 2 and cls in (0, 2)) and not (op == 3 and cls in (0, 1)):
            assert np.abs(ye).max() > 0, (op, cls, interp)


KERNEL = re.compile(r"\b(pv_\w+?_kernel)\b")


def launched(fn):
    """(fn(), the set of this project's kernels the device ran during fn), as test_gpu_dispatch_matrix.launched."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.events():
        if e.device_type == DeviceType.CUDA:
            names |= set(KERNEL.findall(e.name))
    return out, names


def test_routes(drv, eng):
    x = signal()
    _, seen = launched(lambda: chain(drv, x, 1, 1, 0, 0))
    # a time-only stretch expression: sampled per frame, the planned kernel; its lambda: a full table, the general one
    assert "pv_fx_sample_kernel" in seen and "pv_stretch_planned_kernel" in seen and "pv_stretch_kernel" not in seen, seen
    _, seen = launched(lambda: chain(drv, x, 1, 1, 0, 1))
    assert "pv_stretch_kernel" in seen and "pv_stretch_planned_kernel" not in seen, seen
    # a frequency-only repitch expression: one row of positions, the shared kernel
    _, seen = launched(lambda: chain(drv, x, 0, 2, 0, 0))
    assert "pv_repitch_shared_kernel" in seen, seen
    _, seen = launched(lambda: chain(drv, x, 0, 2, 0, 1))
    assert "pv_repitch_shared_kernel" not in seen, seen
    # modify_frequency with an expression stays on the device: both tables from the kernels, the PV never downloaded
    (_, _, host), seen = launched(lambda: chain(drv, x, 3, 3, 0, 0))
    assert "pv_fx_at_pv_kernel" in seen and host == 0
    _, _, host = chain(drv, x, 3, 3, 0, 1)
    assert host == 1, "the lambda route evaluates mod at every MF on the host"


def test_invalid_expressions_give_null_pvs(drv):
    x = noise_chirp(8000, SR, 3).astype(np.float32)
    assert drv.fx_refusals(x.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), x.size, SR) == 1


def test_time_only_stretch_expression_stays_sharded(tmp_path):
    """PV::stretch( fx::curve( fx::t, ... ) ) (a time-only factor between 0.8 and 1.5) through libflan_b200_host.so on a
    PV larger than 256 MB, with one device and with several behind the process-wide engine (on a one-GPU box the device listed three times), each in its own process:
    with several, the second device runs a stretch (kernel kind 6), and PV and samples are the one-device ones bit for bit."""
    import torch
    script = tmp_path / "run.py"
    script.write_text('''
import ctypes, sys, numpy as np
sys.path.insert(0, %r)
from flan_b200 import build, capi
from flan_b200.signals import noise_chirp
L = ctypes.CDLL(build.fx_test_path())
core = capi.load()
multi = ctypes.CDLL(build.host_path())._ZN4flan4b2005multiEv      # flan::b200::multi()
multi.restype = ctypes.c_void_p
m = multi()
second = core.flan_b200_multi_ctx(m, 1) if m else None
fp, ip, i = ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_int), ctypes.c_int
L.fx_chain.argtypes = [fp, i, i, ctypes.c_float, i, i, i, i, i, i, i, fp, ip, fp, ip]
sr, W, h, N, n = 48000.0, 2048, 128, 2048, 4_600_000
x = np.stack([noise_chirp(n, sr, 91)])
F, B = n // h + 1, N // 2 + 1
if second:
    core.flan_b200_set_timing(second, 1)
cap = 2 * F + 16
pv = np.zeros((1, cap, B, 2), np.float32)
y = np.zeros((1, cap * h), np.float32)
frames, host = i(0), i(0)
got = L.fx_chain(x.ctypes.data_as(fp), 1, n, sr, W, h, N, 1, 4, 0, 0, pv.ctypes.data_as(fp), ctypes.byref(frames),
                 y.ctypes.data_as(fp), ctypes.byref(host))
assert got == frames.value * h, (got, frames.value)
probe = -1
if second:
    ms, k = ctypes.c_double(), ctypes.c_int64()
    assert core.flan_b200_kernel_time(second, 6, ctypes.byref(ms), ctypes.byref(k)) == 0
    probe = k.value
np.savez(sys.argv[1], pv[:, :frames.value], y[:, :got], np.array([probe]))
''' % ROOT)
    n_gpus = torch.cuda.device_count()
    results = []
    for env_extra in ({"FLAN_B200_DEVICE": "0"},
                      {"FLAN_B200_DEVICES": ",".join(str(i) for i in range(min(n_gpus, 4))) if n_gpus > 1 else "0,0,0"}):
        env = dict(os.environ)
        env.pop("FLAN_B200_DEVICE", None)
        env.pop("FLAN_B200_DEVICES", None)
        env.update(env_extra)
        path = tmp_path / ("out_%d.npz" % len(results))
        subprocess.run([sys.executable, str(script), str(path)], check=True, env=env, timeout=900)
        results.append(np.load(path))
    one, many = results
    assert one["arr_2"][0] == -1, "FLAN_B200_DEVICE=0 uses one device"
    assert many["arr_2"][0] >= 1, "the stretch ran on the second device: the PV stayed sharded"
    assert one["arr_0"].nbytes > 256 << 20
    for k in ("arr_0", "arr_1"):
        assert one[k].shape == many[k].shape and np.array_equal(bits(one[k]), bits(many[k])), k
    assert np.abs(one["arr_1"]).max() > 0.01
