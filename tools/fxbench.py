"""Expression Functions against lambdas on one config-4 channel (30 min at 48 kHz, W = N = 2048, hop 128).

    python tools/fxbench.py [--seconds 1800] [--reps 3] [--out result.json]

Times PV::repitch, PV::stretch and PV::modify_frequency through the C++ API (tools/cpp/fx_bench.cpp) with a
time-only, a frequency-only and a two-dimensional Function, each written as a lambda (sampled on the host, uploaded)
and as an expression (sampled on the GPU into its compact table), and the constant Function as the floor; each call is
bracketed by a device synchronise, the best of --reps is reported. Then the grid sampler alone
(flan_b200_fx_sample over the full 675001 x 1025 grid) and the at-PV evaluator, with CUDA events, and their rate over
the bytes they store (and read). The card's name and power limit are read in the same run."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=1800.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from flan_b200 import build, capi
    from flan_b200.engine import Engine
    from flan_b200.signals import noise_chirp
    build.build_host()
    sr, W, hop, N = 48000.0, 2048, 128, 2048
    n = int(sr * args.seconds)
    x = noise_chirp(n, sr, 4).astype(np.float32)
    res = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "shape": {"sr": sr, "W": W, "hop": hop, "N": N, "n": n}}

    L = ctypes.CDLL(build.fx_bench_path())
    L.fx_bench_setup.argtypes = [ctypes.POINTER(ctypes.c_float), ctypes.c_int, ctypes.c_float, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    L.fx_bench_call.argtypes = [ctypes.c_int] * 3
    L.fx_bench_call.restype = ctypes.c_double
    F = L.fx_bench_setup(x.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), n, sr, W, hop, N)
    assert F > 0
    B = N // 2 + 1
    res["shape"].update({"frames": F, "bins": B})
    calls = {}
    for op, name in enumerate(["repitch", "stretch", "modify_frequency"]):
        L.fx_bench_call(op, 0, 0)                               # warm-up of the op's kernels
        calls["%s_constant" % name] = min(L.fx_bench_call(op, 0, 0) for _ in range(args.reps))
        for cls, dep in ((1, "t"), (2, "f"), (3, "tf")):
            calls["%s_%s_expression" % (name, dep)] = min(L.fx_bench_call(op, cls, 0) for _ in range(args.reps))
            calls["%s_%s_lambda" % (name, dep)] = L.fx_bench_call(op, cls, 1)
        print(json.dumps({k: round(v, 2) for k, v in calls.items() if k.startswith(name)}), flush=True)
    L.fx_bench_teardown()
    res["call_ms"] = {k: round(v, 3) for k, v in calls.items()}

    eng = Engine(0)
    ts, bw = np.float32(1.0) / np.float32(eng.analysis_rate(sr, hop)), np.float32(sr) / np.float32(N)
    progs = {
        "tf_affine": capi.fx_program(["t", 7200.0, "div", 1.0, "add", "f", 96000.0, "div", "add"]),
        "tf_curve_where": capi.fx_program(["t", 0.5, "mul", "f", 1000.0, "div", "add", "t", "floor", "f", "sqrt", "max", "sub",
                                           "t", 3.0, "lt", ("curve", 0), "f", 9000.0, "gt", "where"],
                                          [([(0.0, 1.0), (1.0, 1.5), (2.0, 0.25)], 5)]),
        "tf_sin": capi.fx_program(["t", 7.0, "mul", "sin", "f", 0.001, "mul", "add"]),
    }
    kern = {}
    for name, prog in progs.items():
        out = eng.fx_sample(prog, F, B, ts, bw)           # warm-up, and the output buffer
        fs, bs = ctypes.c_int64(), ctypes.c_int()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        eng._bind_stream()
        ev[0].record()
        for _ in range(args.reps):
            eng.ctx.call("flan_b200_fx_sample", ctypes.byref(prog), F, B, ts, bw, eng._chk(out), ctypes.byref(fs), ctypes.byref(bs))
        ev[1].record()
        torch.cuda.synchronize()
        ms = ev[0].elapsed_time(ev[1]) / args.reps
        kern["sample_%s" % name] = {"ms": round(ms, 3), "stored_GB": round(out.numel() * 4 / 1e9, 3),
                                    "GB_per_s": round(out.numel() * 4 / ms / 1e6, 1)}
        del out
    pv = torch.empty((1, F, B, 2), dtype=torch.float32, device="cuda")
    pv[..., 1].uniform_(0, 24000)
    pv[..., 0].uniform_(0, 1)
    prog = progs["tf_affine"]
    out = eng.fx_at_pv(prog, pv, np.float32(sr) / np.float32(hop))
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    eng._bind_stream()
    ev[0].record()
    for _ in range(args.reps):
        eng.ctx.call("flan_b200_fx_at_pv", ctypes.byref(prog), eng._chk(pv), 1, F, B, np.float32(sr) / np.float32(hop), eng._chk(out))
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / args.reps
    moved = out.numel() * 4 + pv.numel() * 4          # stores, plus the MF rows it reads
    kern["at_pv_tf_affine"] = {"ms": round(ms, 3), "moved_GB": round(moved / 1e9, 3), "GB_per_s": round(moved / ms / 1e6, 1)}
    res["kernels"] = kern
    print(json.dumps(kern), flush=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
