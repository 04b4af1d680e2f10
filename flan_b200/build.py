"""In-tree builds: libflan_b200.so (nvcc, sm_100a) and the CPU thread emulator used by the tests.

    python -m flan_b200.build          # both

nvcc cross-compiles without a GPU; the .so files are git-ignored but travel to the GPU box with gpurun.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "lib")

NVCC_FLAGS = [
    "-std=c++17", "--expt-relaxed-constexpr",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3",
    "-Xcompiler", "-fPIC,-ffp-contract=off",
]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _sources(*names):
    return [os.path.join(CSRC, n) for n in names]


def lib_path():
    return os.path.join(LIB, "libflan_b200.so")


def emu_path():
    return os.path.join(LIB, "libpv_emu.so")


def debug_lib_path():
    """Development build with the FLAN_B200_* experiment knobs and every kernel variant (tools/experiments)."""
    return os.path.join(LIB, "libflan_b200_debug.so")


def build_library(force=False, verbose=False, debug=False):
    os.makedirs(LIB, exist_ok=True)
    # (source, extra flags): the PV-domain kernels must reproduce the reference's float arithmetic bit for bit, and the
    # expression kernels the host evaluation of flan_b200_fx_eval, so their translation units are compiled without FMA
    # contraction.
    units = [("pv_kernels.cu", []), ("pv_capi.cu", []), ("pv_capi_modify.cu", []), ("pv_capi_io.cu", []),
             ("pv_capi_fx.cu", []), ("pv_modify.cu", ["-fmad=false"]), ("pv_io.cu", ["-fmad=false"]),
             ("pv_fx.cu", ["-fmad=false"])]
    units = [u for u in units if os.path.exists(os.path.join(CSRC, u[0]))]
    for extra_unit in ("pv_generic.cu", "pv_capi_multi.cu", "pv_capi_exchange.cu"):
        if os.path.exists(os.path.join(CSRC, extra_unit)):
            units.append((extra_unit, []))
    srcs = _sources(*[u for u, _ in units])
    deps = srcs + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))] + \
        [os.path.join(os.path.dirname(HERE), "include", "flan_b200.h")]
    target = debug_lib_path() if debug else lib_path()
    if not force and not _newer(target, deps):
        return target
    objdir = os.path.join(LIB, "obj_debug" if debug else "obj")
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for (name, extra), src in zip(units, srcs):
        obj = os.path.join(objdir, name + ".o")
        objs.append(obj)
        cmd = ["nvcc"] + NVCC_FLAGS + extra + (["-DFLAN_B200_DEBUG"] if debug else []) + (["-Xptxas", "-v"] if verbose else []) + \
            ["-c", "-o", obj, src]
        procs.append((cmd, subprocess.Popen(cmd)))
    for cmd, p in procs:
        if p.wait() != 0:
            raise subprocess.CalledProcessError(p.returncode, cmd)
    subprocess.run(["nvcc", "-shared", "-o", target] + objs, check=True)
    return target


def build_emulator(force=False):
    os.makedirs(LIB, exist_ok=True)
    src = os.path.join(CSRC, "emu", "pv_emu.cpp")
    src_modify = os.path.join(CSRC, "emu", "pv_modify_emu.cpp")
    deps = [src, src_modify] + _sources("pv_core.cuh", "pv_body.cuh", "pv_tables.h", "pv_modify_body.cuh", "pv_policy.h", "pv_kernel_list.h",
                                        "pv_generic.h", "pv_generic_body.cuh")
    if not force and not _newer(emu_path(), deps):
        return emu_path()
    cuda_inc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    cmd = ["g++", "-O2", "-ffp-contract=off", "-std=c++20", "-fPIC", "-shared", "-I" + cuda_inc,
           "-o", emu_path(), src, src_modify, "-lpthread"]
    subprocess.run(cmd, check=True)
    return emu_path()


HOST = os.path.join(HERE, "host")


def host_path():
    return os.path.join(LIB, "libflan_b200_host.so")


def api_test_path():
    return os.path.join(LIB, "libflan_api_test.so")


def wav_test_path():
    """tests/cpp/wav_formats_driver.cpp: WAV files of every sample type through flan::Audio::load / save."""
    return os.path.join(LIB, "libflan_wav_test.so")


def fx_test_path():
    """tests/cpp/fx_driver.cpp: expression Functions (flan/fx.h) and their lambdas through the PV-domain methods."""
    return os.path.join(LIB, "libflan_fx_test.so")


def fx_bench_path():
    """tools/cpp/fx_bench.cpp: the PV-domain methods timed with lambdas and expressions (tools/fxbench.py)."""
    return os.path.join(LIB, "libflan_fx_bench.so")


def e2e_bench_path():
    return os.path.join(LIB, "libflan_e2e_bench.so")


def build_host(force=False):
    """The C++ side of the boundary (flan::Audio / flan::PV over the C ABI) and the API test driver."""
    build_library(force)
    os.makedirs(LIB, exist_ok=True)
    root = os.path.dirname(HERE)
    srcs = [os.path.join(HOST, "src", n) for n in ("b200_storage.cpp", "AudioBuffer.cpp", "PVBuffer.cpp", "AudioPV.cpp", "PVModify.cpp", "fx.cpp")]
    hdrs = []
    for d, _, files in os.walk(os.path.join(HOST, "include")):
        hdrs += [os.path.join(d, f) for f in files]
    inc = ["-I" + os.path.join(HOST, "include"), "-I" + os.path.join(root, "include")]
    common = ["g++", "-O2", "-std=c++20", "-fPIC", "-shared", "-Wall"] + inc
    link = ["-L" + LIB, "-Wl,-rpath,$ORIGIN"]
    if force or _newer(host_path(), srcs + hdrs + [lib_path()]):
        subprocess.run(common + ["-o", host_path()] + srcs + link + ["-lflan_b200"], check=True)
    drv = os.path.join(root, "tests", "cpp", "flan_api_driver.cpp")
    if force or _newer(api_test_path(), [drv, host_path()] + hdrs):
        subprocess.run(common + ["-o", api_test_path(), drv] + link + ["-lflan_b200_host", "-lflan_b200"], check=True)
    wav_drv = os.path.join(root, "tests", "cpp", "wav_formats_driver.cpp")
    if os.path.exists(wav_drv) and (force or _newer(wav_test_path(), [wav_drv, host_path()] + hdrs)):
        subprocess.run(common + ["-o", wav_test_path(), wav_drv] + link + ["-lflan_b200_host", "-lflan_b200"], check=True)
    fx_drv = os.path.join(root, "tests", "cpp", "fx_driver.cpp")
    if force or _newer(fx_test_path(), [fx_drv, host_path()] + hdrs):
        subprocess.run(common + ["-o", fx_test_path(), fx_drv] + link + ["-lflan_b200_host", "-lflan_b200"], check=True)
    e2e = os.path.join(root, "tools", "cpp", "e2e_bench.cpp")
    if os.path.exists(e2e) and (force or _newer(e2e_bench_path(), [e2e, host_path()] + hdrs)):
        subprocess.run(common + ["-o", e2e_bench_path(), e2e] + link + ["-lflan_b200_host", "-lflan_b200", "-lpthread"], check=True)
    fxb = os.path.join(root, "tools", "cpp", "fx_bench.cpp")
    if os.path.exists(fxb) and (force or _newer(fx_bench_path(), [fxb, host_path()] + hdrs)):
        subprocess.run(common + ["-o", fx_bench_path(), fxb] + link + ["-lflan_b200_host", "-lflan_b200"], check=True)
    ex = os.path.join(root, "examples", "pv_chain.cpp")
    exe = os.path.join(LIB, "pv_chain")
    if os.path.exists(ex) and (force or _newer(exe, [ex, host_path()] + hdrs)):
        subprocess.run(["g++", "-O2", "-std=c++20", "-Wall"] + inc + ["-o", exe, ex] + link + ["-lflan_b200_host", "-lflan_b200"], check=True)
    return host_path()


def build_all(force=False):
    build_library(force)
    build_emulator(force)
    build_host(force)


if __name__ == "__main__":
    if "--debug" in sys.argv:
        print(build_library(force="--force" in sys.argv, debug=True))
        sys.exit(0)
    build_all(force="--force" in sys.argv)
    print(lib_path())
    print(emu_path())
