"""The PV-domain chain over frame-range shards (flan_b200_multi_repitch / _stretch / _modify_time, pv_capi_multi.cu):
repitch keeps the shards, a bin-shared map that never descends gives a PV sharded for its own frame count, anything else
gathers onto device 0 and gives one shard. Every result must be the single-device result bit for bit, the input must stay
as it was, and the resynthesis of a sharded result must equal the single-device one -- with the promise that the rows
are unchanged, one launch fewer on every device (the stretch left the phase summaries). On a one-GPU box the device is
listed several times, as in test_gpu_multi.py."""
import ctypes

import numpy as np
import pytest

from flan_b200 import capi
from flan_b200.signals import noise_chirp, sine_sweep

pytestmark = pytest.mark.gpu

SR, W, HOP, N = 48000.0, 2048, 128, 2048
B = N // 2 + 1


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


@pytest.fixture(scope="module")
def eng():
    from flan_b200.engine import Engine
    return Engine(0)


class Multi:
    def __init__(self, devices):
        self.lib = capi.load()
        arr = (ctypes.c_int * len(devices))(*devices)
        self.h = ctypes.c_void_p()
        rc = self.lib.flan_b200_multi_create(arr, len(devices), ctypes.byref(self.h))
        assert rc == 0, self.lib.flan_b200_multi_last_error(None)
        self.n = len(devices)

    def call(self, name, *args):
        rc = getattr(self.lib, name)(self.h, *args)
        assert rc == 0, (name, self.lib.flan_b200_multi_last_error(self.h))

    def launches(self):
        return [int(self.lib.flan_b200_launch_count(self.lib.flan_b200_multi_ctx(self.h, i))) for i in range(self.n)]

    def gather(self, pv):
        out = np.empty((pv.channels, pv.frames, pv.bins, 2), np.float32)
        self.call("flan_b200_multi_gather_pv", ctypes.byref(pv), out.ctypes.data, 0, None)
        return out

    def table_call(self, name, pv, table, F):
        """table: a float (constant), [F, B] (full), [B] (row) or [F, 1] (column), host memory."""
        t = np.ascontiguousarray(np.asarray(table, np.float32).reshape(-1) if np.ndim(table) == 0 else table, np.float32)
        fs, bs = {(F, B): (B, 1), (B,): (0, 1), (F, 1): (1, 0)}.get(t.shape, (0, 0))
        out = capi.ShardedPV()
        self.call(name, ctypes.byref(pv), t.ctypes.data, fs, bs, 0, ctypes.byref(out))
        return out

    def resynthesise(self, pv, promise):
        if promise:
            self.call("flan_b200_multi_promise_unchanged", ctypes.byref(pv))
        n0 = self.launches()
        a = capi.ShardedAudio()
        self.call("flan_b200_multi_convert_to_audio", ctypes.byref(pv), ctypes.byref(a))
        y = np.empty((pv.channels, pv.frames * HOP), np.float32)
        self.call("flan_b200_multi_gather_audio", ctypes.byref(a), y.ctypes.data)
        self.call("flan_b200_multi_free_audio", ctypes.byref(a))
        return y, [b - a_ for a_, b in zip(n0, self.launches())]

    def close(self):
        self.lib.flan_b200_multi_destroy(self.h)


def _devices(k):
    import torch
    n = torch.cuda.device_count()
    return list(range(min(n, k))) if n >= 2 else [0] * k


def analysed(m, eng, n, C, seed):
    """(sharded PV, the same PV on cuda:0 from the single-device engine, frames)."""
    import torch
    x = np.stack([noise_chirp(n, SR, seed + c) if c % 2 == 0 else sine_sweep(n, SR) for c in range(C)])
    pv = capi.ShardedPV()
    m.call("flan_b200_multi_convert_to_pv_host", x.ctypes.data, C, n, SR, W, HOP, N, ctypes.byref(pv))
    ref = eng.convert_to_pv(torch.from_numpy(x).cuda(), SR, W, HOP, N)
    return pv, ref, n // HOP + 1


def time_only(F, seed):
    return np.random.default_rng(seed).uniform(0.3, 3.0, (F, 1)).astype(np.float32)


def flat_run_map(F, ar):
    t = np.arange(F, dtype=np.float32)[:, None] / np.float32(ar)
    m = t * np.float32(1.3) + np.float32(0.02)
    m[F // 3:F // 3 + 200] = m[F // 3]                  # a flat run: those pairs cover no output frame
    return np.ascontiguousarray(m, np.float32)


@pytest.mark.parametrize("k", [2, 3, 4])
@pytest.mark.parametrize("case", ["const2", "const05_full_repitch", "time_only", "modify_time_flat"])
def test_sharded_chain_is_bit_identical_to_one_device(eng, k, case):
    import torch
    m = Multi(_devices(k))
    C = 2 if case != "time_only" else 1
    pv, ref, F = analysed(m, eng, 1_500_000, C, 7)
    assert pv.shards > 1
    ar = eng.analysis_rate(SR, HOP)
    before = m.gather(pv)
    assert np.array_equal(bits(before), bits(ref.cpu().numpy()))

    rp_table = np.random.default_rng(1).uniform(0.5, 2.0, (F, B)).astype(np.float32) if case == "const05_full_repitch" else 1.5
    rp = m.table_call("flan_b200_multi_repitch", pv, rp_table, F)
    rp_ref = eng.repitch(ref, SR, torch.from_numpy(rp_table).cuda() if np.ndim(rp_table) else rp_table, 0)
    assert rp.shards == pv.shards and list(rp.frame_begin)[:k + 1] == list(pv.frame_begin)[:k + 1]
    assert np.array_equal(bits(m.gather(rp)), bits(rp_ref.cpu().numpy()))
    assert np.array_equal(bits(m.gather(pv)), bits(before)), "the input PV changed"

    if case == "modify_time_flat":
        table = flat_run_map(F, ar)
        st = m.table_call("flan_b200_multi_modify_time", rp, table, F)
        st_ref = eng.modify_time(rp_ref, SR, ar, torch.from_numpy(table).cuda(), 0)
    else:
        table = {"const2": 2.0, "const05_full_repitch": 0.5, "time_only": time_only(F, 3)}[case]
        st = m.table_call("flan_b200_multi_stretch", rp, table, F)
        st_ref = eng.stretch(rp_ref, SR, ar, torch.from_numpy(table).cuda() if np.ndim(table) else table, 0)
    rp_after = m.gather(rp)
    assert np.array_equal(bits(rp_after), bits(rp_ref.cpu().numpy())), "the input PV changed"
    assert st.frames == st_ref.shape[1] and st.shards > 1
    fb = list(st.frame_begin)[:st.shards + 1]
    assert fb[0] == 0 and fb[-1] == st.frames and all(a < b for a, b in zip(fb, fb[1:]))
    assert np.array_equal(bits(m.gather(st)), bits(st_ref.cpu().numpy()))

    y_ref = eng.convert_to_audio(st_ref, SR, ar, W).cpu().numpy()
    # the first resynthesis on these contexts, with the promise: the summaries the stretch left are used on every device
    # (the stretch reserved the workspace that resynthesis needs, so nothing reallocates it in between) ...
    y_prom, n_prom = m.resynthesise(st, promise=True)
    assert np.array_equal(bits(y_prom), bits(y_ref))
    # ... and without it the rows are read again: one launch more on every device
    y_plain, n_plain = m.resynthesise(st, promise=False)
    assert np.array_equal(bits(y_plain), bits(y_ref))
    assert [a - b for a, b in zip(n_plain, n_prom)][:st.shards] == [1] * st.shards, (n_plain, n_prom)
    for p in (pv, rp, st):
        m.call("flan_b200_multi_free_pv", ctypes.byref(p))
    m.close()


@pytest.mark.parametrize("kind", ["per_bin_stretch", "descending_map"])
def test_other_maps_gather_to_one_shard(eng, kind):
    import torch
    m = Multi(_devices(3))
    pv, ref, F = analysed(m, eng, 600_000, 2, 11)
    assert pv.shards > 1
    ar = eng.analysis_rate(SR, HOP)
    before = m.gather(pv)
    if kind == "per_bin_stretch":
        table = np.random.default_rng(4).uniform(0.5, 2.0, (F, B)).astype(np.float32)
        out = m.table_call("flan_b200_multi_stretch", pv, table, F)
        want = eng.stretch(ref, SR, ar, torch.from_numpy(table).cuda(), 0)
    else:
        t = np.arange(F, dtype=np.float32)[:, None] / np.float32(ar)
        table = np.ascontiguousarray(t[::-1] * np.float32(1.2), np.float32)
        out = m.table_call("flan_b200_multi_modify_time", pv, table, F)
        want = eng.modify_time(ref, SR, ar, torch.from_numpy(table).cuda(), 0)
    assert out.shards == 1 and out.frames == want.shape[1]
    assert np.array_equal(bits(m.gather(out)), bits(want.cpu().numpy()))
    assert np.array_equal(bits(m.gather(pv)), bits(before))
    y, _ = m.resynthesise(out, promise=False)
    assert np.array_equal(bits(y), bits(eng.convert_to_audio(want, SR, ar, W).cpu().numpy()))
    m.call("flan_b200_multi_free_pv", ctypes.byref(out))
    m.call("flan_b200_multi_free_pv", ctypes.byref(pv))
    m.close()


def test_short_signal_uses_fewer_shards_than_devices(eng):
    import torch
    m = Multi(_devices(4))
    pv, ref, F = analysed(m, eng, 25_000, 1, 13)         # 196 frames in, 98 out: a shard needs 2 * ceil(W / hop) = 32
    assert pv.shards == 4
    ar = eng.analysis_rate(SR, HOP)
    st = m.table_call("flan_b200_multi_stretch", pv, 0.5, F)
    want = eng.stretch(ref, SR, ar, 0.5, 0)
    assert 1 <= st.shards < 4 and st.frames == want.shape[1]
    assert np.array_equal(bits(m.gather(st)), bits(want.cpu().numpy()))
    y, _ = m.resynthesise(st, promise=False)
    assert np.array_equal(bits(y), bits(eng.convert_to_audio(want, SR, ar, W).cpu().numpy()))
    m.call("flan_b200_multi_free_pv", ctypes.byref(st))
    m.call("flan_b200_multi_free_pv", ctypes.byref(pv))
    m.close()


def test_cpp_api_chain_stays_sharded(tmp_path):
    """flan::PV::repitch / stretch and PV::convert_to_audio through libflan_b200_host.so on a PV larger than 256 MB, with
    one device and with several behind the process-wide engine ($FLAN_B200_DEVICES; on a one-GPU box the device is listed
    three times): constant factors keep the PV sharded through the chain, a per-bin stretch gathers it; PV and samples
    are the single-device ones bit for bit. Each engine lives in its own process. With several devices, the launches on
    the engine's second device show the route: kind 0 stretches there (kernel kind 6) and its resynthesis takes the
    promise (no phase-summary launch, kind 1); kind 1 repitches there (kind 5) but its per-bin stretch is gathered."""
    import os
    import subprocess
    import sys
    import torch
    script = tmp_path / "run.py"
    script.write_text('''
import ctypes, sys, numpy as np
sys.path.insert(0, %r)
from flan_b200 import build, capi
from flan_b200.signals import noise_chirp
L = ctypes.CDLL(build.api_test_path())
core = capi.load()                                     # the same libflan_b200.so the C++ layer uses
multi = ctypes.CDLL(build.host_path())._ZN4flan4b2005multiEv      # flan::b200::multi()
multi.restype = ctypes.c_void_p
m = multi()
second = core.flan_b200_multi_ctx(m, 1) if m else None
fp, ip = ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_int)
i = ctypes.c_int
L.api_chain.argtypes = [fp, i, i, ctypes.c_float, i, i, i, i, i, fp, ip, fp]
sr, W, h, N, n = 48000.0, 2048, 128, 2048, 4_600_000
x = np.stack([noise_chirp(n, sr, 91)])
F, B = n // h + 1, N // 2 + 1
out, probe = [], []
for kind in (0, 1):
    if second:
        core.flan_b200_set_timing(second, 1)
    cap = 2 * F + 16
    pv = np.zeros((1, cap, B, 2), np.float32)
    frames = i(0)
    y = np.zeros((1, cap * h), np.float32)
    got = L.api_chain(x.ctypes.data_as(fp), 1, n, sr, W, h, N, kind, 0, pv.ctypes.data_as(fp), ctypes.byref(frames), y.ctypes.data_as(fp))
    assert got == frames.value * h, (kind, got, frames.value)
    out += [pv[:, :frames.value], y[:, :got]]
    if second:
        ms, n_launch = ctypes.c_double(), ctypes.c_int64()
        counts = []
        for k in (1, 5, 6):
            assert core.flan_b200_kernel_time(second, k, ctypes.byref(ms), ctypes.byref(n_launch)) == 0
            counts.append(n_launch.value)
        probe.append(counts)
np.save(sys.argv[1] + ".probe.npy", np.array(probe, np.int64).reshape(-1, 3))
np.savez(sys.argv[1], *out)
''' % os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    results, probes = [], []
    n_gpus = torch.cuda.device_count()
    for env_extra in ({"FLAN_B200_DEVICE": "0"}, {"FLAN_B200_DEVICES": ",".join(str(i) for i in range(min(n_gpus, 4))) if n_gpus > 1 else "0,0,0"}):
        env = dict(os.environ)
        env.pop("FLAN_B200_DEVICE", None)
        env.pop("FLAN_B200_DEVICES", None)
        env.update(env_extra)
        path = tmp_path / ("out_%d.npz" % len(results))
        subprocess.run([sys.executable, str(script), str(path)], check=True, env=env, timeout=900)
        results.append(np.load(path))
        probes.append(np.load(str(path) + ".probe.npy"))
    one, many = results
    assert probes[0].size == 0, "FLAN_B200_DEVICE=0 uses one device"
    (seg0, rep0, str0), (_, rep1, str1) = probes[1].tolist()
    assert str0 >= 1 and seg0 == 0, "kind 0: stretched on the second device, resynthesis used the summaries it left"
    assert rep1 >= 1 and str1 == 0, "kind 1: repitched on the second device, the per-bin stretch gathered"
    assert rep0 >= 1
    for k in one.files:
        assert one[k].shape == many[k].shape and np.array_equal(one[k].view(np.uint32), many[k].view(np.uint32)), k
    assert np.abs(one["arr_1"]).max() > 0.01
