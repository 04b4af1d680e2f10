"""The dft-4096 transforms keep their per-frame running state in tensor memory (DESIGN.md 4.1c, 4.3): the analysis that
leaves phase summaries adds its per-bin sums with tcgen05.st instead of red.shared.add, and the standard-shape
resynthesis keeps its overlap-add partials there instead of in a shared-memory ring. Checked on the built library's
SASS when cuobjdump is found; the other dft sizes keep the shared-memory forms."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "flan_b200", "lib", "libflan_b200.so")

ANALYSIS = "_ZN3pvk18pv_analysis_kernelILi%dELi16ELi512ELb1ELb0ELb%dEEEvNS_12AnalysisArgsE"      # dft, EMIT
SYNTH_4096 = "_ZN3pvk26pv_synthesis_mirror_kernelILi4096ELi512ELb1ELb0EEEvNS_9SynthArgsE"


@pytest.fixture(scope="module")
def sass():
    if not os.path.exists(SO):
        pytest.skip("libflan_b200.so is not built")
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not found: the kernels' SASS cannot be read")
    cache = {}

    def get(fn):
        if fn not in cache:
            cache[fn] = subprocess.run([cuobjdump, "-sass", "-fun", fn, SO], capture_output=True, text=True, check=True).stdout
            assert "Function : " + fn in cache[fn], fn
        return cache[fn]
    return get


def ops(text, name):
    """Instructions of one opcode (any modifiers, predicated or not)."""
    return len(re.findall(r"^\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\w+\s+)?" + name + r"[.\s]", text, re.M))


def test_emit_analysis_sums_in_tensor_memory(sass):
    # red.shared.add is ATOMS in SASS; the tensor-memory allocation of both dft-4096 forms issues the same few
    assert ops(sass(ANALYSIS % (4096, 1)), "ATOMS") == ops(sass(ANALYSIS % (4096, 0)), "ATOMS"), \
        "the dft-4096 summary sums still go through shared memory"
    assert ops(sass(ANALYSIS % (4096, 1)), "STTM") > ops(sass(ANALYSIS % (4096, 0)), "STTM")
    for n in (2048, 8192):
        assert ops(sass(ANALYSIS % (n, 1)), "ATOMS") > ops(sass(ANALYSIS % (n, 0)), "ATOMS"), "dft %d keeps the shared-memory sums" % n


def test_resynthesis_partials_in_tensor_memory(sass):
    tm = sass(SYNTH_4096)
    # the tables' and the zeroed partials' four x32 stores, and per frame three x8, one x4 and one x2
    assert ops(tm, "STTM") >= 9
    assert re.search(r"STTM\.x8 ", tm) and re.search(r"STTM\.x4 ", tm) and re.search(r"STTM\.x2 ", tm)
