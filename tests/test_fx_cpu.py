"""Expression Functions on the host (include/flan_b200.h, flan_b200_fx_*): the evaluator the kernels share, against a
numpy float32 restatement of every exact op, the five transcendental ops against Python's double libm rounded to float,
what a program is found to depend on, and the refusal of malformed programs. No GPU needed."""
import ctypes
import math
import os
import re

import numpy as np
import pytest

from flan_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32

SPECIAL = np.array([0.0, -0.0, 1.0, -1.0, 0.5, -0.5, 1.5, -2.5, 0.49999997, 2.5, 3.0, 1e-45, -1e-45, 1.1754942e-38,
                    -5e-39, 1e30, -3e38, 3.4028235e38, 16777217.0, 1e-7, np.inf, -np.inf, np.nan, 7.25, -0.3,
                    1234.5678, 8388609.5], np.float32)


@pytest.fixture(scope="module")
def lib():
    from flan_b200 import build
    build.build_library()
    return capi.load()


def run(lib, prog, t, f):
    out = ctypes.c_float()
    rc = lib.flan_b200_fx_eval(ctypes.byref(prog), float(t), float(f), ctypes.byref(out))
    assert rc == capi.OK, lib.flan_b200_fx_last_error()
    return f32(out.value)


def same(got, want):
    """Bit for bit, except that any NaN matches any NaN (payloads are not part of the contract)."""
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    nan = np.isnan(want)
    return bool(np.array_equal(np.isnan(got), nan) and np.array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32)))


def pairs():
    a = np.repeat(SPECIAL, len(SPECIAL))
    b = np.tile(SPECIAL, len(SPECIAL))
    return a, b


def np_round(x):
    r = np.trunc(x)
    return np.where(np.abs(x - r) >= f32(0.5), r + np.sign(x), r).astype(np.float32)


def np_min(a, b, pick_max=False):
    out = []
    for x, y in zip(a, b):
        if np.isnan(x):
            out.append(y)
        elif np.isnan(y):
            out.append(x)
        elif x == y:
            neg = np.signbit(x)
            out.append((y if neg else x) if pick_max else (x if neg else y))
        else:
            out.append((y if x < y else x) if pick_max else (x if x < y else y))
    return np.array(out, np.float32)


BINARY = {
    "add": lambda a, b: a + b, "sub": lambda a, b: a - b, "mul": lambda a, b: a * b, "div": lambda a, b: a / b,
    "min": np_min, "max": lambda a, b: np_min(a, b, True),
    "lt": lambda a, b: (a < b).astype(np.float32), "le": lambda a, b: (a <= b).astype(np.float32),
    "gt": lambda a, b: (a > b).astype(np.float32), "ge": lambda a, b: (a >= b).astype(np.float32),
    "eq": lambda a, b: (a == b).astype(np.float32), "ne": lambda a, b: (a != b).astype(np.float32),
}
UNARY = {
    "neg": lambda a: -a, "abs": np.abs, "floor": np.floor, "ceil": np.ceil, "round": np_round, "sqrt": np.sqrt,
}


@pytest.mark.parametrize("op", sorted(BINARY))
def test_binary_exact_ops_match_numpy(lib, op):
    a, b = pairs()
    prog = capi.fx_program(["t", "f", op])
    got = [run(lib, prog, x, y) for x, y in zip(a, b)]
    with np.errstate(all="ignore"):
        want = BINARY[op](a, b)
    assert same(got, want), op


@pytest.mark.parametrize("op", sorted(UNARY))
def test_unary_exact_ops_match_numpy(lib, op):
    prog = capi.fx_program(["t", op])
    got = [run(lib, prog, x, 0.0) for x in SPECIAL]
    with np.errstate(all="ignore"):
        want = UNARY[op](SPECIAL).astype(np.float32)
    assert same(got, want), op
    # the same op reading f
    prog_f = capi.fx_program(["f", op])
    assert same([run(lib, prog_f, 0.0, x) for x in SPECIAL], want)


def test_where_and_order_of_operations(lib):
    a, b = pairs()
    prog = capi.fx_program(["t", "t", "f", "where"])            # t != 0 ? t : f
    got = [run(lib, prog, x, y) for x, y in zip(a, b)]
    assert same(got, np.where(a != 0, a, b))
    # (t + 1e8) - 1e8 is evaluated as written: no reassociation, no folding
    prog = capi.fx_program(["t", 1e8, "add", 1e8, "sub"])
    assert run(lib, prog, 1.0, 0.0) == f32(f32(1.0) + f32(1e8)) - f32(1e8) == 0.0
    # t * f + 1: two roundings, no fused multiply-add
    prog = capi.fx_program(["t", "f", "mul", 1.0, "add"])
    x, y = f32(1.0000001), f32(0.99999994)
    assert run(lib, prog, x, y).view(np.uint32) == (x * y + f32(1.0)).view(np.uint32)


def _math(fn, *args):
    try:
        return f32(getattr(math, fn)(*[float(v) for v in args]))
    except (ValueError, OverflowError):
        with np.errstate(all="ignore"):
            return f32(getattr(np, fn if fn != "pow" else "power")(*[np.float64(v) for v in args]))


@pytest.mark.parametrize("fn", ["sin", "cos", "exp", "log"])
def test_transcendental_ops_round_the_double_result(lib, fn):
    xs = np.concatenate([SPECIAL, np.random.default_rng(3).uniform(-60, 60, 400).astype(np.float32)])
    prog = capi.fx_program(["t", fn])
    got = [run(lib, prog, x, 0.0) for x in xs]
    assert same(got, [_math(fn, x) for x in xs]), fn


def test_pow_rounds_the_double_result(lib):
    a, b = pairs()
    prog = capi.fx_program(["t", "f", "pow"])
    got = [run(lib, prog, x, y) for x, y in zip(a, b)]
    assert same(got, [_math("pow", x, y) for x, y in zip(a, b)])


PI, SQRT2 = f32(3.14159274101257324), f32(1.41421353816986084)


def np_interp(i, u):
    u = f32(u)
    return f32({
        0: lambda: u, 1: lambda: f32(0.5), 2: lambda: np_round(np.array([u], np.float32))[0],
        3: lambda: f32(0.0), 4: lambda: f32(1.0),
        5: lambda: u * u * (f32(3.0) - f32(2.0) * u),
        6: lambda: u * u * u * (u * (u * f32(6.0) - f32(15.0)) + f32(10.0)),
        7: lambda: (f32(1.0) - f32(math.cos(float(PI * u)))) / f32(2.0),
        8: lambda: f32(float(SQRT2) * math.sin(float(PI / f32(4.0) * u))),
        9: lambda: np.sqrt(u),
    }[i]())


def np_curve(pts, interp, x):
    xs = [f32(p[0]) for p in pts]
    ys = [f32(p[1]) for p in pts]
    x = f32(x)
    if np.isnan(x):
        return x
    if x <= xs[0]:
        return ys[0]
    if x >= xs[-1]:
        return ys[-1]
    i = max(k for k in range(len(xs) - 1) if xs[k] <= x)
    u = (x - xs[i]) / (xs[i + 1] - xs[i])
    return ys[i] + np_interp(interp, u) * (ys[i + 1] - ys[i])


@pytest.mark.parametrize("interp", range(10))
def test_curve_with_every_named_interpolator(lib, interp):
    pts = [(-1.0, 2.0), (0.0, -0.5), (0.25, 3.0), (1.5, 3.0), (4.0, -7.25)]
    prog = capi.fx_program(["t", ("curve", 0)], [(pts, interp)])
    xs = np.concatenate([SPECIAL, np.linspace(-2, 5, 301, dtype=np.float32), np.array([p[0] for p in pts], np.float32)])
    got = [run(lib, prog, x, 0.0) for x in xs]
    with np.errstate(all="ignore"):
        want = [np_curve(pts, interp, x) for x in xs]
    assert same(got, want), interp
    one = capi.fx_program(["f", ("curve", 0)], [([(3.0, 9.5)], interp)])
    assert [run(lib, one, 0.0, x) for x in (-1.0, 3.0, 5.0)] == [9.5, 9.5, 9.5]


def check(lib, prog):
    ut, uf = ctypes.c_int(-1), ctypes.c_int(-1)
    rc = lib.flan_b200_fx_check(ctypes.byref(prog), ctypes.byref(ut), ctypes.byref(uf))
    return rc, (ut.value, uf.value)


def test_dependence(lib):
    cases = [
        (["t", 20.0, "div", 1.0, "add"], (1, 0)),
        (["f", "sqrt"], (0, 1)),
        ([2.0, 3.0, "pow"], (0, 0)),
        (["t", "f", "lt", 1.0, 2.0, "where"], (1, 1)),
        (["t", 0.0, "mul", "f", "add"], (1, 1)),          # syntactic: t * 0 still reads t
        (["f", ("curve", 0)], (0, 1)),
    ]
    for ops, dep in cases:
        prog = capi.fx_program(ops, [([(0.0, 1.0), (1.0, 2.0)], 0)] if any(isinstance(o, tuple) for o in ops) else [])
        assert check(lib, prog) == (capi.OK, dep), ops


def malformed():
    curve = [([(0.0, 1.0), (1.0, 2.0)], 0)]
    yield "no ops", capi.fx_program([])
    p = capi.fx_program(["t"])
    p.ops = capi.FX_MAX_OPS + 1
    yield "too many ops", p
    p = capi.fx_program(["t", "f", "add"])
    p.op[2].code = 99
    yield "unknown op code", p
    p = capi.fx_program(["t"])
    p.op[0].code = -1
    yield "negative op code", p
    yield "underflow", capi.fx_program(["t", "add"])
    yield "where underflow", capi.fx_program(["t", "f", "where"])
    yield "two results", capi.fx_program(["t", "f"])
    yield "stack too deep", capi.fx_program(["t"] * 17 + ["add"] * 16)
    yield "curve index", capi.fx_program(["t", ("curve", 1)], curve)
    yield "curve without curves", capi.fx_program(["t", ("curve", 0)])
    yield "descending curve", capi.fx_program(["t", ("curve", 0)], [([(1.0, 1.0), (0.0, 2.0)], 0)])
    yield "repeated x", capi.fx_program(["t", ("curve", 0)], [([(1.0, 1.0), (1.0, 2.0)], 0)])
    yield "nan x", capi.fx_program(["t", ("curve", 0)], [([(0.0, 1.0), (math.nan, 2.0)], 0)])
    yield "inf y", capi.fx_program(["t", ("curve", 0)], [([(0.0, math.inf)], 0)])
    yield "bad interpolator", capi.fx_program(["t", ("curve", 0)], [([(0.0, 1.0)], 10)])
    yield "user interpolator", capi.fx_program(["t", ("curve", 0)], [([(0.0, 1.0)], -1)])
    p = capi.fx_program(["t", ("curve", 0)], curve)
    p.curve[0].points = 0
    yield "no points", p
    p.curve[0].points = capi.FX_MAX_POINTS + 1
    yield "too many points", p
    p = capi.fx_program(["t"])
    p.curves = capi.FX_MAX_CURVES + 1
    yield "too many curves", p


@pytest.mark.parametrize("kind,prog", list(malformed()), ids=[k for k, _ in malformed()])
def test_malformed_programs_are_refused(lib, kind, prog):
    rc, _ = check(lib, prog)
    assert rc == capi.INVALID, kind
    assert lib.flan_b200_fx_last_error(), kind
    out = ctypes.c_float()
    assert lib.flan_b200_fx_eval(ctypes.byref(prog), 0.0, 0.0, ctypes.byref(out)) == capi.INVALID
    assert lib.flan_b200_fx_check(None, None, None) == capi.INVALID


def test_nan_results_are_the_canonical_quiet_nan(lib):
    # whatever NaN the arithmetic makes (x86: 0xffc00000 from 0 / 0, a NaN input's own payload), the program returns
    # 0x7fc00000, the NaN the device evaluation returns too
    neg_nan = np.array([0xffc00001], np.uint32).view(np.float32)[0]
    for ops, t, f in ((["t", "f", "div"], 0.0, 0.0), (["t", 1.0, "add"], neg_nan, 0.0), (["t", "sqrt"], -1.0, 0.0),
                      (["t", ("curve", 0)], neg_nan, 0.0), (["t", 1.5, "pow"], -2.0, 0.0), (["t", "log"], -1.0, 0.0)):
        prog = capi.fx_program(ops, [([(0.0, 1.0), (1.0, 2.0)], 0)] if any(isinstance(o, tuple) for o in ops) else [])
        assert run(lib, prog, t, f).view(np.uint32) == 0x7fc00000, ops


def test_deepest_and_longest_programs_are_accepted(lib):
    deep = capi.fx_program(["t"] * 16 + ["add"] * 15)
    assert check(lib, deep) == (capi.OK, (1, 0))
    assert run(lib, deep, 1.5, 0.0) == 24.0
    longest = capi.fx_program(["t"] + [1.0, "add"] * 31 + ["neg"])
    assert longest.ops == capi.FX_MAX_OPS and run(lib, longest, 0.0, 0.0) == -31.0


def test_fx_symbols_are_declared_and_exported(lib):
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "flan_b200.h")).read(), flags=re.S)
    names = {"flan_b200_fx_check", "flan_b200_fx_last_error", "flan_b200_fx_eval", "flan_b200_fx_sample", "flan_b200_fx_at_pv"}
    assert names <= set(re.findall(r"\b(flan_b200_[a-z0-9_]+)\s*\(", text))
    for n in names:
        assert hasattr(lib, n), n
    assert ctypes.sizeof(capi.FxProgram) == 8 + 12 * capi.FX_MAX_OPS + capi.FX_MAX_CURVES * (8 + 8 * capi.FX_MAX_POINTS)


def test_cpp_expressions_evaluate_through_the_library(lib):
    # flan::Function<TF, float>( fx::Expr )::operator() (tests/cpp/fx_driver.cpp: fx_value) is the library's evaluator
    from flan_b200 import build
    build.build_host()
    L = ctypes.CDLL(build.fx_test_path())
    L.fx_value.restype = ctypes.c_float
    L.fx_value.argtypes = [ctypes.c_int] * 3 + [ctypes.c_float] * 2
    t, f = f32(0.0725), f32(3125.0)
    assert L.fx_value(0, 1, 0, t, f) == f32(0.75) + f32(0.5) * t
    assert L.fx_value(1, 2, 0, t, f) == f32(1.0) + f / f32(24000.0)
    assert L.fx_value(3, 3, 0, t, f) == f * (f32(1.0) + t / f32(4.0))
    want = max(f32(0.5), f32(1.0) + f / f32(24000.0) - np.floor(t * f32(4.0)) / f32(8.0) + (f32(0.25) if t < f32(0.05) else f32(0.0)))
    assert L.fx_value(0, 3, 0, t, f) == want
    pts = [(0.0, 1.0), (0.05, 1.5), (0.1, 0.8), (0.2, 1.2)]
    for interp in (0, 5, 6):
        assert same([L.fx_value(0, 4, interp, t, f)], [np_curve(pts, interp, t)])
