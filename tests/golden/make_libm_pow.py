#!/usr/bin/env python
"""Record pow(x, y) of glibc's libm (what CPython's float power calls, so what the reference computes `speed ** exponent`
and `(1 - p0) ** ratio` with) on a seeded sample of the argument families of tests/test_pow_port.py -> libm_pow.npz.

The recording pins include/ppg_pow_tables.h without reading a system library: tests/test_pow_port.py checks that the port
built with those tables reproduces every recorded result bit for bit.  Recorded with glibc 2.39 (x86_64); the libm and its
version are stored in the file.
"""
import ctypes
import ctypes.util
import os
import platform

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
N = 3000  # per family: 8 families x 3000 x 3 float64 stays well under 1 MB


def families(rng, n):
    u = lambda: rng.random(n)  # noqa: E731
    return {
        "speed ** 2": (0.5 + 1.5 * u(), np.full(n, 2.0)),
        "speed ** exponent": (0.5 + 1.5 * u(), 0.5 + 3.0 * u()),
        "(1 - p0) ** ratio": (u() * (1 - 1e-9) + 1e-9, 20.0 * u()),
        "0.4 ** ratio": (np.full(n, 0.4), 50.0 * u()),
        "wide x": (np.ldexp(0.5 + u(), rng.integers(-1000, 1000, n).astype(np.int32)), (u() - 0.5) * 4.0),
        "near over/underflow": (0.5 + u(), (u() - 0.5) * 4000.0),
        "tiny / huge y": (np.ldexp(0.5 + u(), rng.integers(-20, 20, n).astype(np.int32)), np.ldexp(u() - 0.5, rng.integers(-80, 80, n).astype(np.int32))),
        "integer y": (u() * 10 + 1e-12, rng.integers(-20, 21, n).astype(np.float64)),
    }


def main():
    libm_name = ctypes.util.find_library("m")
    libm = ctypes.CDLL(libm_name)
    libm.pow.restype = ctypes.c_double
    libm.pow.argtypes = [ctypes.c_double, ctypes.c_double]
    gnu = ctypes.CDLL(None)
    gnu.gnu_get_libc_version.restype = ctypes.c_char_p
    xs, ys, names = [], [], []
    for name, (x, y) in families(np.random.default_rng(2024), N).items():
        xs.append(np.asarray(x, np.float64))
        ys.append(np.asarray(y, np.float64))
        names += [name] * N
    x, y = np.concatenate(xs), np.concatenate(ys)
    z = np.array([libm.pow(a, b) for a, b in zip(x.tolist(), y.tolist())])
    # every entry of the log table (128 intervals of x's mantissa, glibc e_pow.c log_inline) is exercised
    ix = x.view(np.uint64)
    i = ((ix - np.uint64(0x3FE6955500000000)) >> np.uint64(45)) & np.uint64(127)
    assert len(np.unique(i)) == 128
    out = os.path.join(HERE, "libm_pow.npz")
    np.savez_compressed(out, x=x, y=y, pow=z, family=np.array(names),
                        libm=np.array(f"{libm_name}, glibc {gnu.gnu_get_libc_version().decode()}, {platform.machine()}"))
    print("wrote", out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main()
