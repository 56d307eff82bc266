"""The float64 formatter of the device score writer (sai_b200/csrc/format_double.cuh), host build:
its text equals Python's ``repr(float(x))`` -- and ``str(np.float64(x))``, which the score file's Q and
DD columns are printed with, so that a numpy that prints differently is caught here."""

import ctypes as C
import math

import numpy as np
import pytest


def _texts(values):
    from sai_b200.scoring import format_doubles_host

    raw = format_doubles_host(np.asarray(values, dtype=np.float64))
    return [bytes(r).rstrip(b"\0").decode() for r in raw]


def _check(values):
    values = np.asarray(values, dtype=np.float64)
    got = _texts(values)
    bad = [(repr(float(v)), g) for v, g in zip(values.tolist(), got) if g != repr(float(v))]
    assert not bad, bad[:10]
    bad = [(str(np.float64(v)), g) for v, g in zip(values, got) if g != str(np.float64(v))]
    assert not bad, bad[:10]


def test_random_bit_patterns():
    rng = np.random.default_rng(20261022)
    _check(rng.integers(0, 2**64, size=1_000_000, dtype=np.uint64, endpoint=False).view(np.float64))


def test_unit_interval_and_quantile_lerps():
    rng = np.random.default_rng(7)
    _check(rng.random(1_000_000))
    # np.nanquantile's linear interpolation between neighbouring frequencies, as Q is computed
    lo, hi = rng.random(200_000), rng.random(200_000)
    g = rng.random(200_000)
    _check(lo + (hi - lo) * g)
    k = rng.integers(1, 400, size=200_000)
    _check(np.arange(1, 200_001) % k / k)


def test_special_and_boundary_values():
    _check([0.0, -0.0, math.nan, -math.nan, math.inf, -math.inf, 5e-324, -5e-324, 2.2250738585072014e-308,
            2.225073858507201e-308, 1.7976931348623157e308, -1.7976931348623157e308,
            2.0**53 - 1, 2.0**53, 2.0**53 + 2, float(2**53 + 1), 0.1, 0.2, 0.3, 1 / 3, 2 / 3, 123456789.0, 1.5])
    assert _texts([math.nan, -math.inf, -0.0]) == ["nan", "-inf", "-0.0"]


def test_powers_of_ten_and_neighbours():
    vals = []
    for e in range(-323, 309):
        x = float(f"1e{e}")
        vals += [x, math.nextafter(x, 0.0), math.nextafter(x, math.inf)]
    _check(vals)
    _check([2.0**k for k in range(-1074, 1024)])


def test_layout_boundaries():
    assert _texts([0.0001, 9.999999999999999e-05, 1e16, 9999999999999998.0]) == [
        "0.0001", "9.999999999999999e-05", "1e+16", "9999999999999998.0"]
    _check([0.0001, 9.999999999999999e-05, 1e16, 9999999999999998.0, 1e-5, 12345678901234567.0, 1e22, 1e-7])


@pytest.mark.parametrize("x", [0.5, -1e-300, 1.2345678901234567e-45, 9007199254740993.0, math.inf])
def test_single_value_entry(x):
    from sai_b200 import _cabi

    buf = C.create_string_buffer(32)
    n = _cabi.load().sai_format_double(x, buf)
    assert buf.raw[:n].decode() == repr(float(x))


def test_power_tables_are_generated():
    import subprocess
    import sys
    from pathlib import Path

    gen = Path(__file__).resolve().parent.parent / "tools" / "gen_format_tables.py"
    assert subprocess.run([sys.executable, str(gen), "--check"]).returncode == 0
