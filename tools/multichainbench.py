"""BASELINE config 4's chain behind ONE multi-device handle (flan_b200_multi_*): analysis -> repitch( 1.5 ) ->
stretch( 2.0 ) -> resynthesis with the promise that the stretched rows are unchanged, the PV sharded throughout.

    python tools/multichainbench.py [--seconds S] [--channels C] [--gpus 1,2,4,8] [--steps K] [--check-seconds S]

Per device count: ms per stage (device events: the largest elapsed time of any device, flan_b200_multi_time_*), input
frames/s of the whole chain, and whether the result equals the single-device chain (engine on cuda:0) bit for bit at
--check-seconds, a size where the single-device path fits. Device counts above the visible GPUs are skipped. Prints one
JSON line with the card name and power limit, read in the same run."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from flan_b200 import capi  # noqa: E402
from flan_b200.signals import noise_chirp  # noqa: E402

SR, W, HOP, N = 48000.0, 2048, 128, 2048


class Multi:
    def __init__(self, devices):
        self.lib = capi.load()
        arr = (ctypes.c_int * len(devices))(*devices)
        self.h = ctypes.c_void_p()
        if self.lib.flan_b200_multi_create(arr, len(devices), ctypes.byref(self.h)):
            raise RuntimeError(self.lib.flan_b200_multi_last_error(None))

    def call(self, name, *args):
        rc = getattr(self.lib, name)(self.h, *args)
        if rc:
            raise RuntimeError("%s: %s" % (name, self.lib.flan_b200_multi_last_error(self.h).decode()))

    def timed(self, name, *args):
        self.call("flan_b200_multi_time_begin")
        self.call(name, *args)
        ms = ctypes.c_double()
        self.call("flan_b200_multi_time_end", ctypes.byref(ms))
        return ms.value

    def close(self):
        self.lib.flan_b200_multi_destroy(self.h)


def chain(m, x, times=None):
    """One pass of the chain; returns the samples' sharded descriptor (caller frees) and frees everything else."""
    C, n = x.shape
    a, pv, rp, st, y = capi.ShardedAudio(), capi.ShardedPV(), capi.ShardedPV(), capi.ShardedPV(), capi.ShardedAudio()
    repitch, stretch = np.full(1, 1.5, np.float32), np.full(1, 2.0, np.float32)      # read by the calls below: kept alive
    m.call("flan_b200_multi_scatter_audio", x.ctypes.data, C, n, W, HOP, N, ctypes.byref(a))
    t = {}
    t["analysis"] = m.timed("flan_b200_multi_convert_to_pv", ctypes.byref(a), SR, W, HOP, N, ctypes.byref(pv))
    t["repitch"] = m.timed("flan_b200_multi_repitch", ctypes.byref(pv), repitch.ctypes.data, 0, 0, 0, ctypes.byref(rp))
    t["stretch"] = m.timed("flan_b200_multi_stretch", ctypes.byref(rp), stretch.ctypes.data, 0, 0, 0, ctypes.byref(st))
    m.call("flan_b200_multi_promise_unchanged", ctypes.byref(st))
    t["resynthesis"] = m.timed("flan_b200_multi_convert_to_audio", ctypes.byref(st), ctypes.byref(y))
    shards = st.shards
    for p in (pv, rp, st):
        m.call("flan_b200_multi_free_pv", ctypes.byref(p))
    m.call("flan_b200_multi_free_audio", ctypes.byref(a))
    if times is not None:
        times.append(t)
    return y, shards


def samples(m, y, C, n_out):
    out = np.empty((C, n_out), np.float32)
    m.call("flan_b200_multi_gather_audio", ctypes.byref(y), out.ctypes.data)
    m.call("flan_b200_multi_free_audio", ctypes.byref(y))
    return out


def single_device(x):
    import torch
    from flan_b200.engine import Engine
    eng = Engine(0)
    ar = eng.analysis_rate(SR, HOP)
    pv = eng.convert_to_pv(torch.from_numpy(x).cuda(), SR, W, HOP, N)
    st = eng.stretch(eng.repitch(pv, SR, 1.5, 0), SR, ar, 2.0, 0)
    return eng.convert_to_audio(st, SR, ar, W).cpu().numpy()


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or "unknown (nvidia-smi: %s)" % q.stderr.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=600.0)
    ap.add_argument("--channels", type=int, default=1)
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--check-seconds", type=float, default=60.0)
    args = ap.parse_args()
    import torch
    visible = torch.cuda.device_count()
    if visible < 1:
        raise SystemExit("multichainbench needs a GPU")
    result = {"card": card(), "channels": args.channels, "seconds": args.seconds, "runs": []}
    n = int(SR * args.seconds)
    x = np.stack([noise_chirp(n, SR, 40 + c) for c in range(args.channels)])
    n_chk = int(SR * args.check_seconds)
    x_chk = np.ascontiguousarray(x[:, :n_chk])
    want = single_device(x_chk)
    F = n // HOP + 1
    for g in (int(s) for s in args.gpus.split(",")):
        if g > visible:
            result["runs"].append({"gpus": g, "skipped": "only %d visible" % visible})
            continue
        m = Multi(list(range(g)))
        y, _ = chain(m, x_chk)
        got = samples(m, y, x_chk.shape[0], want.shape[1])
        equal = bool(np.array_equal(got.view(np.uint32), want.view(np.uint32)))
        times = []
        y, _ = chain(m, x)                      # warm-up at the timed size
        m.call("flan_b200_multi_free_audio", ctypes.byref(y))
        shards = 0
        for _ in range(args.steps):
            y, shards = chain(m, x, times)
            m.call("flan_b200_multi_free_audio", ctypes.byref(y))
        m.close()
        ms = {k: float(np.median([t[k] for t in times])) for k in times[0]}
        total = sum(ms.values())
        result["runs"].append({"gpus": g, "ms": ms, "total_ms": total, "input_frames_per_s": F * args.channels / (total / 1e3),
                               "stretched_shards": shards, "bit_equal_to_one_device": equal})
    print(json.dumps(result))


if __name__ == "__main__":
    main()
