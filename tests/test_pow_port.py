"""include/ppg_pow.h — the bit-exact twin of glibc's pow() that the device uses for `speed ** exponent` (ECO:559-563) and
`(1 - p0) ** ratio` (STAG:1137) — against the running libm (what CPython's float power calls): identical bits on millions
of arguments over the reference's domain and far outside of it (over / underflow, tiny and huge exponents)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SRC = r"""
#include <math.h>
#include <stdint.h>
#include <string.h>
#include "ppg_pow.h"
/* number of arguments where the port and libm differ in any bit; first mismatch into bad[2] */
long compare(const double* x, const double* y, long n, double* bad) {
  long k = 0;
  for (long i = 0; i < n; ++i) {
    const double a = pow(x[i], y[i]), c = ppg_pow(x[i], y[i]);
    uint64_t ua, uc; memcpy(&ua, &a, 8); memcpy(&uc, &c, 8);
    if (ua != uc && !(a != a && c != c)) { if (!k) { bad[0] = x[i]; bad[1] = y[i]; } ++k; }
  }
  return k;
}
double one(double x, double y) { return ppg_pow(x, y); }
void many(const double* x, const double* y, long n, double* out) { for (long i = 0; i < n; ++i) out[i] = ppg_pow(x[i], y[i]); }
"""


def _lib(d):
    open(os.path.join(d, "p.c"), "w").write(SRC)
    so = os.path.join(d, "p.so")
    # same floating-point flags as the oracle (no contraction: the port spells its fused operations out)
    subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-I", os.path.join(ROOT, "include"), os.path.join(d, "p.c"), "-o", so, "-lm"])
    L = C.CDLL(so)
    L.compare.restype = C.c_long
    L.compare.argtypes = [C.c_void_p, C.c_void_p, C.c_long, C.c_void_p]
    L.one.restype = C.c_double
    L.one.argtypes = [C.c_double, C.c_double]
    L.many.argtypes = [C.c_void_p, C.c_void_p, C.c_long, C.c_void_p]
    return L


def test_pow_port_is_bit_identical_to_libm():
    rng = np.random.default_rng(7)
    n = 1_000_000
    u = lambda: rng.random(n)  # noqa: E731
    cases = {
        "speed ** 2": (0.5 + 1.5 * u(), np.full(n, 2.0)),
        "speed ** exponent": (0.5 + 1.5 * u(), 0.5 + 3.0 * u()),
        "(1 - p0) ** ratio": (u() * (1 - 1e-9) + 1e-9, 20.0 * u()),
        "0.4 ** ratio": (np.full(n, 0.4), 50.0 * u()),
        "wide x": (np.ldexp(0.5 + u(), rng.integers(-1000, 1000, n).astype(np.int32)), (u() - 0.5) * 4.0),
        "near over/underflow": (0.5 + u(), (u() - 0.5) * 4000.0),
        "tiny / huge y": (np.ldexp(0.5 + u(), rng.integers(-20, 20, n).astype(np.int32)), np.ldexp(u() - 0.5, rng.integers(-80, 80, n).astype(np.int32))),
        "integer y": (u() * 10 + 1e-12, rng.integers(-20, 21, n).astype(np.float64)),
    }
    with tempfile.TemporaryDirectory() as d:
        L = _lib(d)
        for name, (x, y) in cases.items():
            x, y = np.ascontiguousarray(x, np.float64), np.ascontiguousarray(y, np.float64)
            bad = np.zeros(2)
            k = L.compare(x.ctypes.data, y.ctypes.data, n, bad.ctypes.data)
            assert k == 0, f"{name}: {k} of {n} differ, first pow({bad[0].hex()}, {bad[1].hex()})"
        assert L.one(0.4, 0.0) == 1.0 and L.one(1.0, 123.0) == 1.0 and L.one(2.0, 0.5) == 2.0 ** 0.5


def test_pow_tables_are_this_libms():
    """include/ppg_pow_tables.h holds the tables of glibc's pow (written by scripts/extract_glibc_pow_tables.py): the port built
    with them reproduces, bit for bit, pow results recorded from glibc 2.39's libm (tests/golden/libm_pow.npz, made by
    tests/golden/make_libm_pow.py; the sample exercises every entry of the log table)"""
    z = np.load(os.path.join(ROOT, "tests", "golden", "libm_pow.npz"))
    x, y, want = z["x"], z["y"], z["pow"]
    got = np.zeros_like(want)
    with tempfile.TemporaryDirectory() as d:
        _lib(d).many(x.ctypes.data, y.ctypes.data, x.size, got.ctypes.data)
    bad = np.nonzero(got.view(np.uint64) != want.view(np.uint64))[0]
    assert bad.size == 0, [(str(z["family"][i]), x[i].hex(), y[i].hex(), got[i].hex(), want[i].hex()) for i in bad[:3]]
