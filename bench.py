#!/usr/bin/env python
"""bench.py -- PV frames/sec (analysis + resynthesis) of the B200 phase-vocoder engine.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] ...     # the reference's own CPU path (oracle/_ref)

Workload (BASELINE.json configs[1]): stereo 48 kHz, 10 minutes of seeded noise + chirp per GPU, window 4096,
hop 256, dft 4096 -> 112 501 frames x 2 channels x 2049 bins per GPU (3.69 GB of PV data, far larger than the
126 MB L2, so no cache flush is needed between steps). A step is one pass of the hot path over that batch:
Audio::convert_to_PV followed by PV::convert_to_audio, inputs resident in HBM. With N > 1 the signal is N times
as long and frame-range sharded (weak scaling): each rank transforms its contiguous frame range; resynthesis
exchanges the per-bin phase state (all_gather) and the window-hop overlap-add halo (send/recv) over NCCL.

One JSON line on stdout (rank 0). `value` = frames of all ranks / max-over-ranks device time (CUDA events). With
--steps K exactly K steps are timed; without it, rounds of 20 steps (each bracketed by its own events) are repeated until
about --min-seconds of device time has been measured. `ms_per_step` is the mean over all timed steps.
--dump-outputs DIR writes what the last timed step computed (a seeded sample of the PV rows and of the resynthesised
audio, with their indices) as DIR/*.npy, so that two builds can be compared output for output on identical inputs.
`e2e` = the same step through the reference-facing C++ API (tools/cpp/e2e_bench.cpp: flan::Audio holding a host
std::vector -> convert_to_PV -> convert_to_audio -> get_buffer()), host vectors in and out every step, beside the
copy-only ceiling of the same bytes over PCIe.
`roofline` = algorithmic bytes of the dominant kernel / its CUDA-event duration, against MEASURED_PEAKS.json; `roofline_legs`
the same for each leg and for the whole round trip.
`cpu_baseline` = the reference's own sources (oracle/_ref, vendored pffft as the FFTW stand-in), one thread as
written, on a bounded sample of the same signal.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
_REAL_STDOUT = 1


def emit(line):
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())

import numpy as np  # noqa: E402

SR, W, HOP, N_DFT, CH = 48000.0, 4096, 256, 4096, 2
SECONDS_PER_GPU = 600
WORKLOAD = "cfg2: stereo 48 kHz 10 min noise+chirp per GPU, window 4096 hop 256 dft 4096, convert_to_PV + convert_to_audio"
FALLBACK_HBM_GBS = 6650.0
E2E_THREADS = 3


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--seconds", type=float, default=SECONDS_PER_GPU, help="signal length per GPU (debug only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--exchange", choices=["peer", "nccl"], default="peer",
                    help="N > 1: how the phase state and the overlap-add halo travel between the ranks")
    ap.add_argument("--no-summary-hint", action="store_true",
                    help="N = 1: analysis without flan_b200_hint_resynthesis (resynthesis then reads the rows twice, as in round 1)")
    ap.add_argument("--no-cfg3", action="store_true", help="skip the BASELINE config 3 leg (1 h mono 96 kHz through the multi-device handle)")
    ap.add_argument("--min-seconds", type=float, default=1.0, help="without --steps: device time to cover with rounds of 20 steps")
    ap.add_argument("--chain", action="store_true",
                    help="instead of the headline line: BASELINE config 4's chain (analysis -> repitch -> stretch -> resynthesis) "
                         "on one channel per GPU, with the reference's own PVModify.cpp timed beside it")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a seeded sample of what the last timed step computed (PV rows, audio) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.chain or args.impl != "ours"):
        ap.error("--dump-outputs applies to the headline round trip only")
    return args


# ------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock, power and throttle reasons sampled every few ms DURING the timed region (NVML; nvidia-smi as fallback)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.stop = threading.Event()
        self.th = None
        self.nvml = None
        self.handle = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
        except Exception:
            self.nvml = None

    @staticmethod
    def _physical_index(index):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[index])
            except Exception:
                pass
        return index

    def _poll_nvml(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        try:
            rs = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:
            rs = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        pw = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
        self.samples.append({"sm": float(sm), "max": float(mx), "power": pw, "reasons": int(rs)})

    def _poll_smi(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader,nounits", "-i", str(self.index)],
                             capture_output=True, text=True, timeout=10).stdout.strip().splitlines()
        if out:
            f = [x.strip() for x in out[0].split(",")]
            rs = 0
            for bit, val in zip((0x8, 0x40, 0x20, 0x4), f[3:7]):
                if val.lower().startswith("active"):
                    rs |= bit
            self.samples.append({"sm": float(f[0]), "max": float(f[1]), "power": float(f[2]), "reasons": rs})

    def _run(self):
        while not self.stop.is_set():
            try:
                if self.nvml:
                    self._poll_nvml()
                else:
                    self._poll_smi()
            except Exception:
                pass
            self.stop.wait(0.004)

    def __enter__(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=15)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock samples"]}
        sm = sorted(x["sm"] for x in self.samples)
        bits = 0
        for x in self.samples:
            bits |= x["reasons"]
        reasons = [name for bit, name in self.REASONS.items() if bits & bit]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.samples[0]["max"], "reasons": reasons,
                "samples": len(self.samples), "power_w_max": max(x["power"] for x in self.samples),
                "source": "nvml" if self.nvml else "nvidia-smi"}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return FALLBACK_HBM_GBS, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


# ------------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the reference's own sources (oracle/_ref)
# ------------------------------------------------------------------------------------------------------
def cpu_reference_run(seconds, threads, steps, warmup):
    """Round trips of `seconds` of the workload signal per thread, `threads` host threads. Returns frames/s."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_lib import RefLib
    from flan_b200.signals import noise_chirp
    if not RefLib.available():
        raise RuntimeError("oracle/_ref/libflan_ref.so missing (built by __graft_entry__.build() where /root/reference exists)")
    ref = RefLib(1)      # vendored pffft as the FFTW stand-in: the reference's float-SIMD speed class
    n = int(SR * seconds)
    chunks = [np.stack([noise_chirp(n, SR, 1234 + i)]) for i in range(threads)]
    frames_per_chunk = n // HOP + 1

    def work(i):
        ref.bench(chunks[i], SR, W, HOP, N_DFT, 1)

    def step():
        th = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
        for t in th:
            t.start()
        for t in th:
            t.join()

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return frames_per_chunk * threads * steps / dt, dt / steps, frames_per_chunk * threads


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps if args.steps is not None else 3
    warmup = args.warmup if args.warmup is not None else 1
    cores = os.cpu_count() or 1
    seconds = 30.0
    try:
        fps, step_s, frames = cpu_reference_run(seconds, cores, steps, warmup)
    except Exception as e:  # the oracle always exists; this is a broken checkout
        emit({"impl": "reference", "unavailable": str(e)})
        return
    sample = "%d host threads x one mono %g s chunk of the cfg2 signal each per step (%d frames/step), reference " \
             "AudioPV.cpp compiled verbatim, FFTW stand-in = vendored pffft" % (cores, seconds, frames)
    line = {
        "impl": "reference",
        "metric": "PV frames/sec (analysis+resynth)", "value": fps, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": step_s * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------------
# our arm

def copy_only_ceiling(torch, dev, nbytes_up, nbytes_down, steps):
    """Seconds per step of moving one step's input up and one step's output down over PCIe and nothing else: pinned
    buffers, two streams, both directions at once (what a perfectly overlapped pipeline would be left with)."""
    up_h = torch.empty(nbytes_up, dtype=torch.uint8).pin_memory()
    dn_h = torch.empty(nbytes_down, dtype=torch.uint8).pin_memory()
    up_d = torch.empty(nbytes_up, dtype=torch.uint8, device=dev)
    dn_d = torch.empty(nbytes_down, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def go(k):
        for _ in range(k):
            with torch.cuda.stream(s1):
                up_d.copy_(up_h, non_blocking=True)
            with torch.cuda.stream(s2):
                dn_h.copy_(dn_d, non_blocking=True)
        s1.synchronize()
        s2.synchronize()

    go(2)
    t0 = time.perf_counter()
    go(steps)
    return (time.perf_counter() - t0) / steps


DUMP_FRAMES, DUMP_SAMPLES, DUMP_SEED = 1024, 1 << 20, 20240601


def dump_outputs(torch, outdir, pv, audio):
    """The last timed step's outputs, as a caller receives them: PV rows (C, frames, bins, 2) and audio (C, n). A fixed,
    seeded sample of at most DUMP_FRAMES rows and DUMP_SAMPLES audio samples per channel is written, with the indices it
    was taken at (with the default workload: 3.69 GB of PV, about 50 MB written)."""
    os.makedirs(outdir, exist_ok=True)
    rng = np.random.default_rng(DUMP_SEED)
    frames = np.sort(rng.choice(pv.shape[1], min(DUMP_FRAMES, pv.shape[1]), replace=False))
    samples = np.sort(rng.choice(audio.shape[1], min(DUMP_SAMPLES, audio.shape[1]), replace=False))
    pick = lambda t, idx: t.index_select(1, torch.from_numpy(idx).to(t.device)).cpu().numpy()  # noqa: E731
    out = {"pv_frames": frames.astype(np.float64), "pv": pick(pv, frames).astype(np.float32),
           "audio_samples": samples.astype(np.float64), "audio": pick(audio, samples).astype(np.float32)}
    for name, a in out.items():
        np.save(os.path.join(outdir, name + ".npy"), a)


def cfg3_leg(world, steps, peak):
    """BASELINE config 3 (mono 96 kHz 1 h, window 8192 hop 512, round trip) through the multi-device handle of the C ABI
    (flan_b200_multi_*: one process, frame-range shards, P2P phase-state + halo exchange): on one device and, when the run
    has several GPUs, on all of them -- the strong-scaling figure. Inputs resident in HBM, device-timed (max over devices)."""
    import ctypes
    from flan_b200 import capi
    from flan_b200.signals import noise_chirp
    lib = capi.load()
    sr, w, hop, n_dft = 96000.0, 8192, 512, 8192
    n = int(sr * 3600)
    chunk = noise_chirp(int(sr * 60), sr, 3)
    x = np.ascontiguousarray(np.tile(chunk, 60)[None, :n])
    F, B = n // hop + 1, n_dft // 2 + 1
    byts = 2.0 * (4.0 * n + 8.0 * F * B)                 # SURVEY 8d: read + write once per direction
    out = {"workload": "cfg3: mono 96 kHz 1 h, window 8192 hop 512 dft 8192, round trip, frame-range shards cut at segment "
                       "boundaries, phase state + overlap-add halo exchanged device to device (flan_b200_multi_*)", "frames": F}
    for k in sorted({1, world}):
        devs = (ctypes.c_int * k)(*range(k))
        h = ctypes.c_void_p()
        if lib.flan_b200_multi_create(devs, k, ctypes.byref(h)) != 0:
            out["gpus_%d" % k] = {"error": lib.flan_b200_multi_last_error(None).decode()}
            continue

        def call(name, *a):
            rc = getattr(lib, name)(h, *a)
            if rc != 0:
                raise RuntimeError("%s: %s" % (name, lib.flan_b200_multi_last_error(h).decode()))
        a = capi.ShardedAudio()
        call("flan_b200_multi_scatter_audio", x.ctypes.data, 1, n, w, hop, n_dft, ctypes.byref(a))

        def step():
            pv, y = capi.ShardedPV(), capi.ShardedAudio()
            call("flan_b200_multi_hint_resynthesis")          # a round trip: the shards' analysis leaves their phase summaries
            call("flan_b200_multi_convert_to_pv", ctypes.byref(a), sr, w, hop, n_dft, ctypes.byref(pv))
            call("flan_b200_multi_promise_unchanged", ctypes.byref(pv))
            call("flan_b200_multi_convert_to_audio", ctypes.byref(pv), ctypes.byref(y))
            call("flan_b200_multi_free_pv", ctypes.byref(pv))
            call("flan_b200_multi_free_audio", ctypes.byref(y))
        for _ in range(3):
            step()
        ms = ctypes.c_double(0)
        call("flan_b200_multi_time_begin")
        for _ in range(steps):
            step()
        call("flan_b200_multi_time_end", ctypes.byref(ms))
        t = ms.value / steps
        out["gpus_%d" % k] = {"ms_per_round_trip": t, "frames_per_s": F / (t * 1e-3), "shards": int(a.shards),
                              "hbm_gbs_per_gpu": byts / k / (t * 1e-3) / 1e9, "frac_of_peak_per_gpu": byts / k / (t * 1e-3) / 1e9 / peak}
        call("flan_b200_multi_free_audio", ctypes.byref(a))
        lib.flan_b200_multi_destroy(h)
    if world > 1 and "frames_per_s" in out.get("gpus_1", {}) and "frames_per_s" in out.get("gpus_%d" % world, {}):
        out["strong_scaling_speedup"] = out["gpus_%d" % world]["frames_per_s"] / out["gpus_1"]["frames_per_s"]
    return out


def e2e_cpp(args, local_rank, world, rank, steps, dist, dev):
    import ctypes
    import torch
    from flan_b200 import build
    from flan_b200.signals import noise_chirp
    os.environ["FLAN_B200_DEVICE"] = str(local_rank)      # the C++ layer's process-wide context
    # built by build(); the benchmark compiles nothing, so it can run from a read-only tree
    if not os.path.exists(build.e2e_bench_path()):
        raise RuntimeError("%s is missing: run `python -m flan_b200.build`" % build.e2e_bench_path())
    L = ctypes.CDLL(build.e2e_bench_path())
    L.e2e_round_trips.restype = ctypes.c_double
    L.e2e_round_trips.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_float, ctypes.c_int, ctypes.c_int,
                                  ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_double)]
    n = int(SR * args.seconds)
    audio = np.stack([noise_chirp(n, SR, 1234 + c + 100 * rank) for c in range(CH)])
    F = n // HOP + 1
    chk = ctypes.c_double(0)

    def run(threads, k, warm):
        if dist is not None:
            dist.barrier()
        dt = L.e2e_round_trips(audio.ctypes.data, CH, n, SR, W, HOP, N_DFT, threads, warm, k, ctypes.byref(chk))
        if dt < 0:
            raise RuntimeError("the C++ API returned a null object in the e2e leg")
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return world * threads * k * CH * F / float(t.item())

    k = steps
    many = run(E2E_THREADS, k, 6)     # 6 untimed passes: by then the host vectors are recycled and page-locked
    two = run(2, k, 6)
    one = run(1, k, 6)
    if dist is not None:
        dist.barrier()                   # every rank measures its copies at the same time, as they run in the e2e leg
    ceil_s = copy_only_ceiling(torch, dev, 4 * CH * n, 4 * CH * F * HOP, k)
    tc = torch.tensor([ceil_s], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(tc, op=dist.ReduceOp.MAX)
    ceiling = world * CH * F / float(tc.item())
    return {"value": many, "unit": "frames/s", "h2d_bytes_per_step": int(4 * CH * n), "d2h_bytes_per_step": int(4 * CH * F * HOP),
            "host_threads": E2E_THREADS, "two_thread_value": two, "single_thread_value": one, "steps_per_thread": k,
            "copy_only_ceiling": ceiling, "frac_of_copy_ceiling": many / ceiling,
            "how": "tools/cpp/e2e_bench.cpp, user code against the reference-facing C++ API: flan::Audio (host std::vector, touched through "
                   "get_buffer() every step) -> convert_to_PV -> convert_to_audio -> get_buffer() on the result; %d host threads on independent "
                   "signals, as a program working through a batch of files would (two_thread_value / single_thread_value: fewer threads); "
                   "copy_only_ceiling = the same bytes up and down over PCIe from cudaHostAlloc'ed memory, both directions at once, nothing "
                   "else (the API's vectors are page-locked with cudaHostRegister; profiles/r2_e2e_timeline.md shows the copies slowing each "
                   "other down: a download slice takes 1.0 ms alone and 1.45 ms beside an upload)" % E2E_THREADS
                   + ("; every rank converts its own signal on its own GPU" if world > 1 else "")}

# ------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from flan_b200.engine import Engine
    from flan_b200.signals import noise_chirp
    from flan_b200.sharding import PeerExchange, frame_shard, sharded_resynthesis_overlapped, sharded_resynthesis_peer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    steps = args.steps if args.steps is not None else 20
    warmup = max(3, args.warmup if args.warmup is not None else 3)
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    # A CPU-side group for the waits during which rank 0 works alone on EVERY GPU (the config 3 leg): an NCCL barrier is a
    # kernel spinning on the waiting ranks' GPUs, which rank 0's process would then have to time-slice with
    # (measured: 33.5 ms per round trip on 2 GPUs beside such a barrier, 7.5 ms without it).
    cpu_group = dist.new_group(backend="gloo") if world > 1 else None
    eng = Engine(local_rank)
    dev = eng.device

    n_total = int(SR * args.seconds) * world
    sh = frame_shard(n_total, HOP, W, world, rank)
    B = N_DFT // 2 + 1
    ar = eng.analysis_rate(SR, HOP)
    n_local = sh.audio_hi - sh.audio_lo
    host_audio = torch.empty((CH, n_local), dtype=torch.float32).pin_memory()
    for c in range(CH):
        host_audio[c].copy_(torch.from_numpy(noise_chirp(n_local, SR, 1234 + c + 100 * rank)))
    x = host_audio.to(dev, non_blocking=True)
    pv = torch.empty((CH, sh.frames, B, 2), dtype=torch.float32, device=dev)
    out_len = sh.span_hi - sh.span_lo
    y = torch.empty((CH, out_len), dtype=torch.float32, device=dev)

    def allgather(state):
        if world == 1:
            return state.unsqueeze(0)
        bufs = torch.empty((world,) + tuple(state.shape), dtype=state.dtype, device=dev)
        dist.all_gather_into_tensor(bufs, state.contiguous())
        return bufs

    hint = not args.no_summary_hint
    side_stream = torch.cuda.Stream(device=dev)
    head_event = torch.cuda.Event()
    head_event.record()                      # creates the handle the C ABI records on
    # The two exchanges of sharded resynthesis (phase state, overlap-add halo) go through flan_b200_exchange_*: peer copies
    # into CUDA-IPC mailboxes ordered by sequence flags (no NCCL kernel beside the transforms). --exchange nccl keeps the
    # torch.distributed form (all_gather + batched send / recv on a side stream).
    exchange, exchange_note = None, None
    if world > 1 and args.exchange == "peer":
        try:
            exchange = PeerExchange(eng, dist, rank, world, CH, B, max(0, W - HOP))
        except RuntimeError as e:      # raised on every rank together: the NCCL form takes over
            exchange_note = str(e)
            if rank == 0:
                print("bench.py: %s; falling back to --exchange nccl" % e, file=sys.stderr)

    def step(xin, yout=None):
        if world == 1:
            # the round trip resynthesises the rows as analysis wrote them: with the hint the analysis kernel also leaves their
            # phase summaries (flan_b200_hint_resynthesis) and resynthesis does not read the rows a second time
            yout = y if yout is None else yout
            eng.convert_to_pv(xin, SR, W, HOP, N_DFT, out=pv, for_resynthesis=hint)
            eng.convert_to_audio(pv, SR, ar, W, out=yout, unchanged=hint)
            return yout
        eng.convert_to_pv_range(xin, sh.audio_lo, n_total, SR, W, HOP, N_DFT, sh.f0, sh.f1, out=pv, for_resynthesis=hint and exchange is not None)
        if exchange is not None:
            o, _ = sharded_resynthesis_peer(eng, exchange, torch, sh, pv, SR, ar, head_event, unchanged=hint)
        else:
            o, _ = sharded_resynthesis_overlapped(eng, dist, torch, sh, pv, SR, ar, allgather, side_stream, head_event)
        return o

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        step(x)
    barrier()

    # ---- timed region: device-resident inputs, CUDA events on the launching stream -----------------------
    # --steps K: one round of exactly K steps. Otherwise K = 20 steps per round, and rounds are repeated until ~1 s of
    # device time is covered so that the clock sampler sees the kernels under load (20 x 3.9 ms gave it one sample).
    eng.set_timing(True)
    rounds = 1
    if args.steps is None:
        for k in eng.KERNEL_KINDS:
            eng.kernel_time(k)
        probe0, probe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        probe0.record()
        step(x)
        probe1.record()
        barrier()
        est = torch.tensor([probe0.elapsed_time(probe1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(est, op=dist.ReduceOp.MAX)
        rounds = int(max(1, min(200, np.ceil(args.min_seconds * 1e3 / max(float(est.item()) * steps, 1e-3)))))
    for k in eng.KERNEL_KINDS:
        eng.kernel_time(k)
    launches0 = eng.launch_count()
    round_ms = []
    with ClockSampler(local_rank) as clocks:
        for _ in range(rounds):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            e0.record()
            for _ in range(steps):
                last = step(x)
            e1.record()
            barrier()
            round_ms.append(e0.elapsed_time(e1))
    launches = (eng.launch_count() - launches0) // rounds
    ktimes = {k: eng.kernel_time(k) for k in eng.KERNEL_KINDS}
    eng.set_timing(False)
    if args.dump_outputs is not None and rank == 0:      # N > 1: rank 0's frame range and audio span
        dump_outputs(torch, args.dump_outputs, pv, last)
    del last
    # for comparison (N = 1): the same round trip without the hint -- analysis as a caller who keeps the PV for something
    # else runs it, resynthesis with its own pass over the rows for the phase summaries (round 1's form)
    plain_ms, plain_kernels = None, None
    if world == 1 and hint:
        hint = False
        for _ in range(3):
            step(x)
        torch.cuda.synchronize()
        eng.set_timing(True)
        for k in eng.KERNEL_KINDS:
            eng.kernel_time(k)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step(x)
        e1.record()
        torch.cuda.synchronize()
        plain_ms = e0.elapsed_time(e1) / steps
        pk = {k: eng.kernel_time(k) for k in ("analysis", "phase_seg", "phase_scan", "synthesis")}
        plain_kernels = {k: (v[0] / v[1] if v[1] else None) for k, v in pk.items()}
        eng.set_timing(False)
        hint = True
    t = torch.tensor(round_ms, dtype=torch.float64, device=dev)
    rank_ms = [float(t.mean().item()) / steps]           # every rank's own mean step (diagnostic: which rank is the slowest)
    if world > 1:
        mine = torch.tensor(rank_ms, dtype=torch.float64, device=dev)
        every = torch.empty((world,), dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(every, mine)
        rank_ms = [float(v) for v in every.tolist()]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)         # per round: the slowest rank
    ms_max = float(t.mean().item())                      # mean round, K steps each
    ms = ms_max
    frames_rank = CH * sh.frames
    frames_all = torch.tensor([frames_rank], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(frames_all, op=dist.ReduceOp.SUM)
    frames_all = float(frames_all.item())
    value = frames_all * steps / (ms_max * 1e-3)

    # ---- end to end: through the reference-facing C++ API, host std::vector in, host std::vector out, every step ----
    # tools/cpp/e2e_bench.cpp is user code against flan::Audio / flan::PV: each step the Audio's host vector is the newest
    # copy (the upload happens inside convert_to_PV), and get_buffer() on the result brings the samples back. Two host
    # threads convert independent signals at the same time, as a program working through a batch of files would, so
    # one thread's download overlaps the other's upload (PCIe is full duplex); the single-thread figure is reported too.
    # With N > 1 every rank converts its own signal of the per-GPU shape on its own GPU (no exchange on this leg).
    del pv, y, x
    torch.cuda.empty_cache()
    e2e = e2e_cpp(args, local_rank, world, rank, steps, dist if world > 1 else None, dev)
    # BASELINE config 3 on rank 0, through the one-process multi-device handle (the other ranks wait at the barrier below)
    cfg3 = None
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier(group=cpu_group)        # every rank's GPU is idle from here on
    if rank == 0 and not args.no_cfg3:
        try:
            cfg3 = cfg3_leg(world, steps, measured_peak()[0])
        except Exception as e:  # noqa: BLE001 - a leg must not take the headline line down with it
            cfg3 = {"error": repr(e)}
    if rank == 0:
        peak, peak_src = measured_peak()
        an_ms, an_n = ktimes["analysis"]
        sy_ms, sy_n = ktimes["synthesis"]
        seg_ms, seg_n = ktimes["phase_seg"]
        scan_ms, scan_n = ktimes["phase_scan"]
        an_bytes = 4.0 * CH * n_local + 8.0 * CH * sh.frames * B          # per launch: audio read + PV written
        sy_bytes = 8.0 * CH * sh.frames * B + 4.0 * CH * out_len          # per launch: PV read + audio written
        kern = []
        if an_n and hint and (world == 1 or exchange is not None):
            # the instantiation that also writes the phase summaries of its rows (32 bytes per bin and segment of <= 128 frames)
            segs = -(-sh.frames // 127)
            kern.append(("pv_analysis_kernel<4096> +summaries", an_bytes + 32.0 * CH * segs * B, an_ms / an_n))
        elif an_n:
            kern.append(("pv_analysis_kernel<4096>", an_bytes, an_ms / an_n))
        if sy_n:
            kern.append(("pv_synthesis_mirror_kernel<4096>", sy_bytes, sy_ms / sy_n))
        dom = max(kern, key=lambda k: k[2]) if kern else None
        roofline = None
        try:        # dram__bytes_read.sum + dram__bytes_write.sum per launch of the same kernel on the same workload (ncu)
            traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))["kernels"]
        except Exception:
            traffic = {}
        if dom:
            ach = dom[1] / (dom[2] * 1e-3) / 1e9
            tr = traffic.get(dom[0], {}) if (world == 1 and args.seconds == SECONDS_PER_GPU) else {}
            roofline = {"bound": "hbm", "kernel": dom[0], "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                        "traffic": tr.get("dram_bytes_per_launch"), "traffic_capture": tr.get("capture"),
                        "peak_source": peak_src, "algorithmic_bytes_per_launch": dom[1], "ms_per_launch": dom[2]}
        per_kernel = {}
        for name, byts, m in kern:
            per_kernel[name] = {"ms_per_launch": m, "achieved_gbs": byts / (m * 1e-3) / 1e9, "frac": byts / (m * 1e-3) / 1e9 / peak}
        if seg_n:
            per_kernel["pv_phase_seg_kernel"] = {"ms_per_launch": seg_ms / seg_n}
        if scan_n:
            per_kernel["pv_phase_scan_kernel"] = {"ms_per_launch": scan_ms / scan_n}
        # the whole round trip against its compulsory traffic 2 * (4h + 8B) bytes per frame (SURVEY.md 8d)
        rt_bytes = (an_bytes + sy_bytes) * steps
        step_gbs = rt_bytes / (ms * 1e-3) / 1e9

        def leg(byts, m):
            return {"ms": m, "algorithmic_bytes": byts, "achieved_gbs": byts / (m * 1e-3) / 1e9, "frac": byts / (m * 1e-3) / 1e9 / peak} if m else None
        legs_roofline = {
            "analysis (pv_analysis_kernel)": leg(an_bytes, an_ms / an_n if an_n else 0),
            "resynthesis kernel (pv_synthesis_mirror_kernel)": leg(sy_bytes, sy_ms / sy_n if sy_n else 0),
            "resynthesis leg (phase summary + scan + kernel)": leg(sy_bytes, (sy_ms + seg_ms + scan_ms) / sy_n if sy_n else 0),
            "round trip (one step)": leg(an_bytes + sy_bytes, ms / steps),
            "peak_gbs": peak, "peak_source": peak_src}
        line = {
            "metric": "PV frames/sec (analysis+resynth)", "value": value, "unit": "frames/s",
            "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms_max / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "channels": CH, "frames_per_gpu": sh.frames, "bins": B,
                       "seconds_per_gpu": args.seconds, "sharding": "none" if world == 1 else "contiguous frame ranges, dp%d; phase state + halo exchange: %s" % (
                           world, "peer copies into CUDA-IPC mailboxes (flan_b200_exchange_*)" if exchange is not None else "NCCL all_gather + send/recv" + (
                               " (%s)" % exchange_note if exchange_note else "")),
                       "l2": "inputs larger than L2 (3.69 GB PV per GPU), no flush",
                       "phase_summaries": ("left by the analysis kernel (flan_b200_hint_resynthesis): the round trip resynthesises the rows unchanged"
                                           if (hint and (world == 1 or exchange is not None)) else "second pass over the rows (pv_phase_seg_kernel)")},
            # analysis-only throughput (BASELINE config 2's wording): the PV is the product there, so the PLAIN kernel counts --
            # timed in the comparison loop when the main loop ran the instantiation that also leaves the phase summaries
            "legs": {"analysis_frames_per_s": (frames_rank / (plain_kernels["analysis"] * 1e-3) if (plain_kernels and plain_kernels.get("analysis"))
                                               else (frames_rank / (an_ms / an_n * 1e-3) if an_n else None)),
                     "analysis_with_summaries_frames_per_s": (frames_rank / (an_ms / an_n * 1e-3) if (an_n and plain_kernels) else None),
                     "resynthesis_frames_per_s": frames_rank / ((sy_ms + seg_ms + scan_ms) / sy_n * 1e-3) if sy_n else None,
                     "audio_samples_per_s": value * HOP,
                     "round_trip_hbm_gbs": step_gbs, "round_trip_frac_of_peak": step_gbs / peak},
            "roofline": roofline, "kernels": per_kernel,
            "e2e": e2e, "rounds": rounds, "timed_seconds": sum(round_ms) * 1e-3,
            "roofline_legs": legs_roofline,
            "cfg3_strong": cfg3, "ms_per_step_by_rank": rank_ms, "without_summary_hint": None if plain_ms is None else {
                "ms_per_step": plain_ms, "value": frames_all / (plain_ms * 1e-3), "ms_per_launch": plain_kernels,
                "note": "the same round trip when the analysis does not know that its rows will be resynthesised unchanged: "
                        "the plain analysis kernel, and pv_phase_seg_kernel reads the rows a second time"},
            "gpu_launches": int(launches),
            "clocks": clocks.summary(),
        }
        if world == 1 and not args.no_cpu_baseline:
            try:
                secs = 60.0
                fps, step_s, frames = cpu_reference_run(secs, 1, 1, 0)
                line["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": 1, "kind": "reference",
                                        "sample": "one mono %g s chunk of the cfg2 signal (%d frames), round trip, reference sources "
                                                  "compiled verbatim, FFTW stand-in = vendored pffft, 1 thread as the reference runs" % (secs, frames)}
            except Exception as e:
                line["cpu_baseline"] = {"value": None, "unit": "frames/s", "cores": 0, "kind": "reference", "sample": "unavailable: %s" % e}
        emit(line)
    if world > 1:
        dist.barrier(group=cpu_group)
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------
# secondary line: BASELINE config 4's PV-domain chain (python bench.py --chain)
# ------------------------------------------------------------------------------------------------------
def run_chain(args):
    import torch
    from flan_b200.engine import Engine
    from flan_b200.signals import noise_chirp
    sr, w, hop, n_dft = 48000.0, 2048, 128, 2048
    steps = args.steps if args.steps is not None else 10
    warmup = max(3, args.warmup if args.warmup is not None else 3)
    eng = Engine(0)
    n = int(sr * 1800)                                   # one of config 4's eight channels: 30 min at 48 kHz
    x = torch.from_numpy(np.stack([noise_chirp(n, sr, 40)])).cuda()
    F, B = eng.num_frames(n, hop), n_dft // 2 + 1
    ar = eng.analysis_rate(sr, hop)
    pv = torch.empty((1, F, B, 2), device="cuda")
    rp = torch.empty_like(pv)

    def step():
        eng.convert_to_pv(x, sr, w, hop, n_dft, out=pv)
        eng.repitch(pv, sr, 1.5, 0, out=rp)
        st = eng.stretch(rp, sr, ar, 2.0, 0, summary_window=w)      # also leaves the phase summaries of its rows
        return st.shape[1], eng.convert_to_audio(st, sr, ar, w, unchanged=True)

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    eng.set_timing(True)
    for k in eng.KERNEL_KINDS:
        eng.kernel_time(k)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(0) as clocks:
        e0.record()
        for _ in range(steps):
            F2, _y = step()
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    kt = {k: eng.kernel_time(k)[0] / steps for k in eng.KERNEL_KINDS}
    peak, peak_src = measured_peak()
    row = 8.0 * B
    stage_bytes = {"analysis": 4.0 * n + row * F, "repitch": 2 * row * F, "stretch": row * F + row * F2,
                   "synthesis": row * F2 + 4.0 * F2 * hop}
    line = {"metric": "PV frames/sec (analysis + repitch + stretch + resynth, config 4 chain)", "value": F / (ms * 1e-3),
            "unit": "input frames/s", "n_gpus": 1, "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "cfg4, one channel per GPU: 48 kHz 30 min noise+chirp, window 2048 hop 128, convert_to_PV -> "
                                   "repitch(1.5) -> stretch(2.0) -> convert_to_audio, PV data resident in HBM throughout",
                       "frames_in": F, "frames_out": F2, "bins": B},
            "kernels": {k: {"ms_per_step": v, "achieved_gbs": stage_bytes[k] / (v * 1e-3) / 1e9 if k in stage_bytes and v else None,
                            "frac": stage_bytes[k] / (v * 1e-3) / 1e9 / peak if k in stage_bytes and v else None} for k, v in kt.items()},
            "peak_source": peak_src, "clocks": clocks.summary()}
    if not args.no_cpu_baseline:
        try:        # the reference's own PVModify.cpp (oracle/_ref/libflan_ref_modify.so) on a bounded sample of the same PV data
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            from oracle_lib import RefModifyLib
            ref = RefModifyLib()
            frames = 4000
            sample = np.ascontiguousarray(pv[:, 1000:1000 + frames].cpu().numpy())
            t0 = time.perf_counter()
            r = ref.repitch(sample, sr, ar, w, np.full((frames, B), 1.5, np.float32), 0)
            ref.stretch(r, sr, ar, w, np.full((frames, B), 2.0, np.float32), 0)
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": frames / dt, "unit": "input frames/s (PV::repitch + PV::stretch only)", "cores": 1, "kind": "reference",
                                    "sample": "%d frames of the same PV data through the reference's PV/PVModify.cpp compiled verbatim, "
                                              "one thread (no TBB here: its par_unseq loops run serially); the GPU's repitch + stretch "
                                              "stages take %.3f ms for %d frames" % (frames, kt["repitch"] + kt["stretch"], F),
                                    "gpu_same_stages_frames_per_s": F / ((kt["repitch"] + kt["stretch"]) * 1e-3)}
        except Exception as e:
            line["cpu_baseline"] = {"value": None, "sample": "unavailable: %s" % e}
    emit(line)


def main():
    # Only the JSON line may reach stdout: libraries (NCCL prints its version there) are diverted to stderr.
    global _REAL_STDOUT
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.chain:
        run_chain(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
