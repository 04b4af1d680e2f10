"""Device WAV sample codecs and WAV file I/O, per sample type.

    python tools/wavbench.py [--channels 8] [--samples 86400000] [--reps 10] [--file-mb 1024] [--out profiles/wavbench.json]
                             [--baseline-lib another/libflan_b200.so]

Codecs: flan_b200_pcm_encode / _decode on config 4's audio (8 channels x 86.4 M samples, 2.8 GB of floats: larger than
L2), timed with CUDA events over --reps launches after a warm-up. Bytes moved are computed from shapes, C * n * (4 + width),
and reported as GB/s and as a share of the HBM figure bench.py uses (MEASURED_PEAKS.json when present, else its 6.65 TB/s
fallback). A device-to-device copy of the float buffer is timed the same way as the copy rate the codecs can be held to.
--baseline-lib: another build of the library (an earlier version, say), whose flan_b200_pcm24_encode / _decode are timed
in the same run on the same buffers, and whose bytes are compared with this build's.

Files: save_wav_as and load_wav of a file of about --file-mb MB in a temporary directory, next to plain writes and reads
of the same bytes from Python (one write / readinto call each, i.e. fwrite / fread). The reads come from the page cache
(the file was just written), so they show the host-side cost, not the disk's. Prints a table and one JSON line with the
card name and power limit, read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from flan_b200 import capi  # noqa: E402
from flan_b200.engine import Engine  # noqa: E402

NAMES = {capi.WAV_PCM_U8: "PCM_U8", capi.WAV_PCM_16: "PCM_16", capi.WAV_PCM_24: "PCM_24", capi.WAV_PCM_32: "PCM_32",
         capi.WAV_FLOAT: "FLOAT", capi.WAV_DOUBLE: "DOUBLE"}
FALLBACK_HBM_GBS = 6650.0          # bench.py's figure when MEASURED_PEAKS.json is absent


def hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json"
    except Exception:
        return FALLBACK_HBM_GBS, "bench.py fallback"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or "unknown (nvidia-smi: %s)" % q.stderr.strip()


def event_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def baseline_pcm24(path, audio, data, back, reps):
    """(encode ms, decode ms, same bytes and bits) of flan_b200_pcm24_* of another build, through plain ctypes (its
    symbol list may differ from capi.SYMBOLS)."""
    import ctypes
    lib = ctypes.CDLL(os.path.abspath(path))
    vp = ctypes.c_void_p
    lib.flan_b200_create.argtypes = [ctypes.c_int, ctypes.POINTER(vp)]
    lib.flan_b200_set_stream.argtypes = [vp, vp]
    for name in ("flan_b200_pcm24_encode", "flan_b200_pcm24_decode"):
        getattr(lib, name).argtypes = [vp, vp, ctypes.c_int, ctypes.c_int64, vp]
    h = vp()
    assert lib.flan_b200_create(0, ctypes.byref(h)) == 0
    assert lib.flan_b200_set_stream(h, vp(torch.cuda.current_stream().cuda_stream)) == 0
    C, n = audio.shape
    ours_bytes, ours_back = data.clone(), back.clone()
    enc = event_ms(lambda: lib.flan_b200_pcm24_encode(h, vp(audio.data_ptr()), C, n, vp(data.data_ptr())), reps)
    dec = event_ms(lambda: lib.flan_b200_pcm24_decode(h, vp(data.data_ptr()), C, n, vp(back.data_ptr())), reps)
    same = bool(torch.equal(ours_bytes, data)) and bool(torch.equal(ours_back.view(torch.int32), back.view(torch.int32)))
    return enc, dec, same


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--channels", type=int, default=8)
    ap.add_argument("--samples", type=int, default=86_400_000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--file-mb", type=int, default=1024)
    ap.add_argument("--out", default=None)
    ap.add_argument("--baseline-lib", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("wavbench needs a CUDA device")
    eng = Engine(0)
    peak, peak_src = hbm_peak()
    C, n = args.channels, args.samples
    g = torch.Generator(device="cuda").manual_seed(1)
    audio = (torch.rand((C, n), device="cuda", generator=g) * 2.2 - 1.1).contiguous()
    back = torch.empty_like(audio)
    rows = []
    copy_ms = event_ms(lambda: back.copy_(audio), args.reps)
    copy_gbs = 2 * audio.numel() * 4 / (copy_ms * 1e-3) / 1e9
    print("card: %s   HBM figure %.0f GB/s (%s)" % (card(), peak, peak_src))
    print("%d ch x %d samples; device copy of the floats: %.3f ms, %.0f GB/s" % (C, n, copy_ms, copy_gbs))
    print("%-7s %-6s %9s %9s %8s %9s" % ("type", "dir", "ms", "GB/s", "of HBM", "of copy"))
    for t in (capi.WAV_PCM_U8, capi.WAV_PCM_16, capi.WAV_PCM_24, capi.WAV_PCM_32, capi.WAV_FLOAT, capi.WAV_DOUBLE):
        width = capi.WAV_WIDTH[t]
        data = torch.empty((C * n * width,), dtype=torch.uint8, device="cuda")
        pa, pd = eng._chk(audio), eng._chk(data, torch.uint8)
        pb = eng._chk(back)
        eng._bind_stream()
        enc = event_ms(lambda: eng.ctx.call("flan_b200_pcm_encode", pa, C, n, t, pd), args.reps)
        dec = event_ms(lambda: eng.ctx.call("flan_b200_pcm_decode", pd, C, n, t, pb), args.reps)
        byts = C * n * (4 + width)
        for d, ms in (("encode", enc), ("decode", dec)):
            gbs = byts / (ms * 1e-3) / 1e9
            rows.append({"type": NAMES[t], "dir": d, "ms": ms, "bytes": byts, "gbs": gbs, "frac_of_hbm": gbs / peak,
                         "frac_of_copy": gbs / copy_gbs})
            print("%-7s %-6s %9.3f %9.0f %7.1f%% %8.1f%%" % (NAMES[t], d, ms, gbs, 100 * gbs / peak, 100 * gbs / copy_gbs))
        if t == capi.WAV_PCM_24 and args.baseline_lib:
            benc, bdec, same = baseline_pcm24(args.baseline_lib, audio, data, back, args.reps)
            for d, ms in (("encode", benc), ("decode", bdec)):
                gbs = byts / (ms * 1e-3) / 1e9
                rows.append({"type": "PCM_24 baseline", "dir": d, "ms": ms, "bytes": byts, "gbs": gbs,
                             "frac_of_hbm": gbs / peak, "frac_of_copy": gbs / copy_gbs, "same_result": same})
                print("%-7s %-6s %9.3f %9.0f %7.1f%% %8.1f%%   (baseline build; same bytes and bits: %s)" % (
                    "PCM_24", d, ms, gbs, 100 * gbs / peak, 100 * gbs / copy_gbs, same))
        del data

    # stereo files of about --file-mb MB each: frames per type
    files = []
    print("%-7s %9s %10s %10s %10s %10s" % ("file", "MB", "save ms", "fwrite ms", "load ms", "fread ms"))
    with tempfile.TemporaryDirectory() as tmp:
        for t in (capi.WAV_PCM_16, capi.WAV_PCM_24, capi.WAV_FLOAT, capi.WAV_DOUBLE):
            width = capi.WAV_WIDTH[t]
            frames = (args.file_mb << 20) // (2 * width)
            x = torch.rand((2, frames), device="cuda", generator=g) * 2.2 - 1.1
            path, raw = os.path.join(tmp, "w.wav"), os.path.join(tmp, "raw.bin")
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            eng.save_wav(path, x, 48000.0, t)
            t1 = time.perf_counter()
            y, _ = eng.load_wav(path)
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            assert y.shape == x.shape
            buf = np.empty(2 * frames * width, np.uint8)
            t3 = time.perf_counter()
            with open(raw, "wb") as f:
                f.write(memoryview(buf))
            t4 = time.perf_counter()
            with open(raw, "rb") as f:
                f.readinto(memoryview(buf))
            t5 = time.perf_counter()
            mb = buf.size / 1e6
            files.append({"type": NAMES[t], "mb": mb, "save_ms": (t1 - t0) * 1e3, "load_ms": (t2 - t1) * 1e3,
                          "fwrite_ms": (t4 - t3) * 1e3, "fread_ms": (t5 - t4) * 1e3})
            print("%-7s %9.0f %10.1f %10.1f %10.1f %10.1f" % (NAMES[t], mb, (t1 - t0) * 1e3, (t4 - t3) * 1e3,
                                                               (t2 - t1) * 1e3, (t5 - t4) * 1e3))
            os.remove(path)
            os.remove(raw)
            del y
    result = {"card": card(), "hbm_gbs_figure": peak, "hbm_figure_source": peak_src, "channels": C, "samples": n,
              "reps": args.reps, "copy_ms": copy_ms, "copy_gbs": copy_gbs, "codecs": rows, "files": files}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
