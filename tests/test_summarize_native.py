"""Host-only hooks of `report -s` (nb200_summary_cell_type, nb200_float_repr; DESIGN.md §2.13) against Python's own
int(), float() and repr() on seeded inputs.  No GPU needed."""
import ctypes as ct
import math
import random
import struct

import numpy as np
import pytest

from nimble_b200 import _lib, frontend


@pytest.fixture(scope="module")
def L():
    try:
        return _lib.load()
    except (ImportError, OSError) as e:
        pytest.skip("library not built: %s" % e)


def _python_type(v):
    """What frontend._infer_column makes of one cell on its own: 0 NA, 1 int, 2 float, 3 string (ASCII cells)."""
    if v in frontend._PANDAS_NA:
        return 0, 0.0
    try:
        x = int(v)
        if v.strip() == v and "_" not in v:
            try:
                return 1, float(x)
            except OverflowError:                     # where the Python path raises, the native one gives +-inf
                return 1, -math.inf if x < 0 else math.inf
    except ValueError:
        pass
    if "_" not in v:
        try:
            return 2, float(v)
        except ValueError:
            pass
    return 3, 0.0


def _native_type(L, v):
    b = v.encode()
    d = ct.c_double()
    return L.nb200_summary_cell_type(b, len(b), ct.byref(d)), d.value


def _same_float(a, b):
    return (math.isnan(a) and math.isnan(b)) or (a == b and math.copysign(1, a) == math.copysign(1, b))


def _cells(rng, n):
    pieces = ["0", "1", "9", "00", "12", ".", "e", "E", "+", "-", "_", " ", "\x0b", "\x0c", "\x1c", "\x1f", "inf", "nan",
              "infinity", "INF", "NaN", "x", "5", "e-", "e+3", "1e308", "1e-320", "\"", "#", "N/A"]
    out = list(frontend._PANDAS_NA) + ["5.", ".5", "-.5e-3", "1e400", "-1e400", "1e-400", "00012", "+0", "-0", "1_0",
                                       " 7 ", "7\x1c", "0x1p3", "1e", "--1", "9" * 40, "-" + "9" * 400, "Infinity", "+nan"]
    for _ in range(n):
        out.append("".join(rng.choice(pieces) for _ in range(rng.randrange(1, 5))))
    return out


def test_cell_type_matches_python(L):
    rng = random.Random(5)
    for v in _cells(rng, 30000):
        want = _python_type(v)
        got = _native_type(L, v)
        assert got[0] == want[0], repr(v)
        if want[0] in (1, 2):
            assert _same_float(got[1], want[1]), (repr(v), got[1], want[1])


def test_random_decimal_strings_parse_like_python(L):
    rng = random.Random(6)
    for _ in range(100000):
        v = "%s%s.%se%d" % (rng.choice(["", "-", "+"]), rng.randrange(0, 10 ** rng.randrange(1, 20)),
                            rng.randrange(0, 10 ** rng.randrange(1, 20)), rng.randrange(-330, 320))
        k, d = _native_type(L, v)
        assert k == 2 and _same_float(d, float(v)), v


def _repr(L, x):
    buf = ct.create_string_buffer(64)
    n = L.nb200_float_repr(x, buf, 64)
    assert n > 0
    return buf.value.decode()


def test_float_repr_fixed_points(L):
    for x in [0.0, -0.0, 1.0, 90.0, 1e16, 1e15, 1e-5, 1e-4, 0.0001234, 123456789012345678.0, 1.5e300, 5e-324, -2.5,
              float("inf"), float("-inf"), float("nan"), 0.1, 1 / 3, 2.0 ** 63, 1e22, 9999999999999998.0]:
        assert _repr(L, x) == repr(x)


def test_float_repr_random_doubles(L):
    """A few million random doubles: uniform bit patterns (every exponent) and values near the format switches."""
    rng = np.random.default_rng(8)
    bits = rng.integers(0, 2 ** 63, 2_000_000, dtype=np.int64).astype(np.uint64) | (rng.integers(0, 2, 2_000_000).astype(np.uint64) << np.uint64(63))
    xs = bits.view(np.float64)
    near = np.concatenate([rng.uniform(1e-6, 1e-3, 300_000), rng.uniform(1e14, 1e18, 300_000), rng.integers(0, 10 ** 6, 200_000) * 1.0])
    buf = ct.create_string_buffer(64)
    f = L.nb200_float_repr
    for x in np.concatenate([xs, near]).tolist():
        n = f(x, buf, 64)
        assert buf.raw[:n].decode() == repr(x), x


def test_float_repr_refuses_a_short_buffer(L):
    buf = ct.create_string_buffer(4)
    assert L.nb200_float_repr(1.5e300, buf, 4) == _lib.EINVAL
    assert L.nb200_float_repr(struct.unpack("<d", struct.pack("<Q", 1))[0], None, 0) == _lib.EINVAL
