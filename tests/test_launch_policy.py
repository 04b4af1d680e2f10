"""The launch policy of the transforms (flan_b200/csrc/pv_policy.h: choose_analysis / choose_synthesis) and the release
kernel list (pv_kernel_list.h), without a GPU.

- Every row of tests/test_gpu_dispatch_matrix.py maps to the kernel name that file expects, plus the policy's edges.
- Every kernel of the release list is reached by at least one row, and every row reaches a listed kernel.
- The transform kernels compiled into libflan_b200.so are exactly the release list."""
import ctypes
import os
import re
import shutil
import subprocess

import pytest

from emu_lib import ROOT, Emu

SMS = 148           # a B200's SMs: the dft-2048 frame threshold is C * F >= SMS * 128
HINTED_F = max(6000, SMS * 64 + 1)


def analysis_a(N):
    return "pv_analysis_kernel<%d,8,768,false,false,false>" % N


def analysis_b(N, pad=False, emit=False):
    return "pv_analysis_kernel<%d,16,512,true,%s,%s>" % (N, str(pad).lower(), str(emit).lower())


def synthesis_mirror(N, tps, one, gen):
    return "pv_synthesis_mirror_kernel<%d,%d,%s,%s>" % (N, tps, str(one).lower(), str(gen).lower())


def synthesis_plain(N, tps, one):
    return "pv_synthesis_kernel<%d,%d,%s>" % (N, tps, str(one).lower())


# (W, hop, N, C, whole-signal frames per channel, aligned2, emit wanted, expected kernel)
ANALYSIS_ROWS = [
    # test_analysis_8_points: 300 hops of signal
    (256, 16, 256, 3, 301, True, False, analysis_a(256)),
    (300, 7, 512, 2, 301, False, False, analysis_a(512)),
    (1000, 100, 1024, 3, 301, True, False, analysis_a(1024)),
    # test_analysis_2048_large_switch, and the threshold in C * F with C = 1
    (2048, 128, 2048, 1, SMS * 128 - 1, True, False, analysis_a(2048)),
    (2048, 128, 2048, 1, SMS * 128, True, False, analysis_b(2048)),
    # test_analysis_mirror_1024
    (1024, 64, 1024, 3, 301, True, False, "pv_analysis_mirror_kernel<1024,512>"),
    # test_analysis_16_points: 200 hops of signal
    (4096, 256, 4096, 2, 201, True, False, analysis_b(4096)),
    (3000, 100, 4096, 3, 201, True, False, analysis_b(4096)),
    (4096, 255, 4096, 2, 201, False, False, analysis_b(4096)),
    (4096, 512, 4096, 3, 201, True, False, analysis_b(4096)),
    (4096, 4096, 4096, 2, 201, True, False, analysis_b(4096)),
    (64, 16, 4096, 3, 201, True, False, analysis_b(4096)),
    (8192, 512, 8192, 2, 201, True, False, analysis_b(8192)),
    (5000, 300, 8192, 3, 201, True, False, analysis_b(8192)),
    # test_analysis_padded_window
    (2048, 128, 4096, 2, 200, True, False, analysis_b(4096, pad=True)),
    (768, 96, 4096, 3, 200, True, False, analysis_b(4096, pad=True)),
    (256, 400, 4096, 2, 200, True, False, analysis_b(4096, pad=True)),
    (4096, 512, 8192, 2, 200, True, False, analysis_b(8192, pad=True)),
    (1024, 64, 2048, 2, SMS * 64, True, False, analysis_b(2048, pad=True)),
    # test_analysis_misaligned_input_leaves_the_padded_form: the input one float past an 8-byte boundary
    (2048, 128, 4096, 3, 201, False, False, analysis_b(4096)),
    # test_hinted_analysis_leaves_summaries: two channels of HINTED_F frames, hinted and plain
    (4096, 256, 4096, 2, HINTED_F, True, True, analysis_b(4096, emit=True)),
    (4096, 128, 4096, 2, HINTED_F, True, True, analysis_b(4096, emit=True)),
    (4096, 200, 4096, 2, HINTED_F, True, True, analysis_b(4096, emit=True)),
    (8192, 512, 8192, 2, HINTED_F, True, True, analysis_b(8192, emit=True)),
    (2048, 128, 2048, 2, HINTED_F, True, True, analysis_b(2048, emit=True)),
    (4096, 256, 4096, 2, HINTED_F, True, False, analysis_b(4096)),
    (2048, 128, 2048, 2, HINTED_F, True, False, analysis_b(2048)),
    # the summaries are refused where that kernel does not apply: W < N, dft 1024, dft 2048 below the frame threshold
    (2048, 128, 4096, 2, HINTED_F, True, True, analysis_b(4096, pad=True)),
    (3000, 100, 4096, 2, HINTED_F, True, True, analysis_b(4096)),
    (1024, 64, 1024, 2, HINTED_F, True, True, "pv_analysis_mirror_kernel<1024,512>"),
    (2048, 128, 2048, 1, SMS * 128 - 1, True, True, analysis_a(2048)),
    # dft 2048 and 4096 at the standard shape take no mirrored analysis
    (2048, 128, 2048, 1, 301, True, False, analysis_a(2048)),
    # a size without a templated kernel
    (1000, 100, 1000, 2, 301, True, False, "pv_generic_analysis_kernel"),
]

# (W, hop, N, expected kernel)
SYNTHESIS_ROWS = [
    # test_synthesis_4096_standard_shape_variants
    (4096, 256, 4096, synthesis_mirror(4096, 512, True, False)),
    # test_synthesis
    (1024, 64, 1024, synthesis_mirror(1024, 384, False, False)),
    (2048, 128, 2048, synthesis_mirror(2048, 384, False, False)),
    (2048, 128, 4096, synthesis_mirror(4096, 384, False, True)),
    (3072, 96, 4096, synthesis_mirror(4096, 384, False, True)),
    (4096, 128, 4096, synthesis_mirror(4096, 384, False, True)),
    (4096, 130, 4096, synthesis_mirror(4096, 384, False, True)),
    (256, 2, 4096, synthesis_mirror(4096, 384, False, True)),
    (1024, 64, 2048, synthesis_mirror(2048, 384, False, True)),
    (512, 32, 1024, synthesis_mirror(1024, 384, False, True)),
    (8192, 512, 8192, synthesis_mirror(8192, 512, True, False)),
    (4096, 256, 8192, synthesis_mirror(8192, 512, True, True)),
    (8192, 1024, 8192, synthesis_plain(8192, 1024, True)),
    (8192, 511, 8192, synthesis_plain(8192, 1024, True)),
    (4096, 255, 4096, synthesis_plain(4096, 768, False)),
    (4096, 512, 4096, synthesis_plain(4096, 768, False)),
    (3000, 100, 4096, synthesis_plain(4096, 768, False)),
    (256, 16, 256, synthesis_plain(256, 768, False)),
    (300, 7, 512, synthesis_plain(512, 768, False)),
    (1000, 50, 1024, synthesis_plain(1024, 768, False)),
    (2048, 127, 2048, synthesis_plain(2048, 768, False)),
    # edges: a hop above one slot, a size without a templated kernel
    (2048, 256, 2048, synthesis_plain(2048, 768, False)),
    (1000, 100, 1000, "pv_generic_synthesis_kernel"),
]


@pytest.fixture(scope="module")
def lib():
    from flan_b200 import build
    build.build_emulator()
    L = Emu().L
    L.pv_emu_choose_analysis.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.c_int,
                                         ctypes.c_int, ctypes.c_int, ctypes.c_char_p, ctypes.c_int]
    L.pv_emu_choose_synthesis.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_char_p, ctypes.c_int]
    L.pv_emu_release_kernels.argtypes = [ctypes.c_char_p, ctypes.c_int]
    return L


def call_name(fn, *args):
    buf = ctypes.create_string_buffer(1 << 14)
    n = fn(*args, buf, len(buf))
    assert n >= 0
    return buf.value.decode()


def choose_analysis(lib, W, hop, N, C, frames, aligned2, emit):
    return call_name(lib.pv_emu_choose_analysis, N, W, hop, C, frames, SMS, int(aligned2), int(emit))


def choose_synthesis(lib, W, hop, N):
    return call_name(lib.pv_emu_choose_synthesis, N, W, hop)


def release_list(lib):
    names = call_name(lib.pv_emu_release_kernels).split()
    assert len(names) == len(set(names))
    return set(names)


@pytest.mark.parametrize("W,hop,N,C,frames,aligned2,emit,expect", ANALYSIS_ROWS)
def test_analysis_rows(lib, W, hop, N, C, frames, aligned2, emit, expect):
    assert choose_analysis(lib, W, hop, N, C, frames, aligned2, emit) == expect


@pytest.mark.parametrize("W,hop,N,expect", SYNTHESIS_ROWS)
def test_synthesis_rows(lib, W, hop, N, expect):
    assert choose_synthesis(lib, W, hop, N) == expect


def test_rows_reach_exactly_the_release_list(lib):
    """Every release kernel is reached by a row (no instantiation without a shape that selects it), and every row's
    templated kernel is in the list (the policy returns nothing the library does not carry)."""
    reached = {r[-1] for r in ANALYSIS_ROWS + SYNTHESIS_ROWS if "generic" not in r[-1]}
    listed = release_list(lib)
    assert not listed - reached, "listed kernels no row reaches: %s" % sorted(listed - reached)
    assert not reached - listed, "rows reach kernels outside the list: %s" % sorted(reached - listed)
    assert len(listed) == 28


MANGLED = re.compile(r"Function : _ZN3pvk\d+(pv_(?:analysis|synthesis)\w*_kernel)I((?:L[ib]\d+E)+)EEv")


def library_kernels(path, cuobjdump):
    """Normalised names of the pv_analysis* / pv_synthesis* kernels in a library's SASS."""
    sass = subprocess.run([cuobjdump, "-sass", path], capture_output=True, text=True, check=True).stdout
    out = set()
    for kind, args in MANGLED.findall(sass):
        vals = [("true" if v == "1" else "false") if t == "b" else v for t, v in re.findall(r"L([ib])(\d+)E", args)]
        out.add("%s<%s>" % (kind, ",".join(vals)))
    return out


def test_library_carries_exactly_the_release_list(lib):
    so = os.path.join(ROOT, "flan_b200", "lib", "libflan_b200.so")
    if not os.path.exists(so):
        pytest.skip("libflan_b200.so is not built")
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not found: the library's kernels cannot be listed")
    built = library_kernels(so, cuobjdump)
    listed = release_list(lib)
    assert built == listed, "built but not listed: %s; listed but not built: %s" % (sorted(built - listed), sorted(listed - built))
