"""CPU tests of the shortest round-trip double formatter (fslr_b200/csrc/fmt_double.cuh) that renders the
`avg_alignment_score` column of mappings.representative.bed on the device: its host build must give exactly Python's
repr(float), which is what pandas' DataFrame.to_csv writes for a float64 column."""
import ctypes
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "tests", "_build")
SLOT = 32


def _lib():
    os.makedirs(BUILD, exist_ok=True)
    so = os.path.join(BUILD, "libhost_fmt_double.so")
    deps = [os.path.join(ROOT, "tests", "host_fmt_double_harness.cpp"), os.path.join(ROOT, "fslr_b200", "csrc", "fmt_double.cuh")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["g++", "-O2", "-shared", "-fPIC", "-x", "c++", "-o", so, deps[0]])
    lib = ctypes.CDLL(so)
    lib.host_fmt_many.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p, ctypes.c_void_p]
    lib.host_fmt_many.restype = None
    return lib


def _check(values):
    x = np.ascontiguousarray(values, dtype=np.float64)
    out = np.zeros(x.shape[0] * SLOT, np.uint8)
    ln = np.zeros(x.shape[0], np.int32)
    _lib().host_fmt_many(x.ctypes.data, x.shape[0], out.ctypes.data, ln.ctypes.data)
    assert ln.min(initial=1) > 0 and ln.max(initial=0) <= 24
    slots = out.reshape(-1, SLOT)
    got = [slots[i, :ln[i]].tobytes().decode() for i in range(x.shape[0])]
    want = [repr(v) for v in x.tolist()]
    if got != want:
        i = next(i for i in range(len(got)) if got[i] != want[i])
        raise AssertionError("value %r (bits %016x): formatter gave %r" % (want[i], x[i:i + 1].view(np.uint64)[0], got[i]))


def test_random_bit_patterns():
    rng = np.random.default_rng(11)
    u = rng.integers(0, 2**64, 1_000_000, dtype=np.uint64, endpoint=False)
    u[::5] &= np.uint64((1 << 63) | ((1 << 52) - 1))                   # a fifth subnormal (exponent field 0), both signs
    x = u.view(np.float64)
    _check(x[np.isfinite(x)])


def test_mean_domain_grid():
    """s / c as the representative file computes it: an integer score sum over a read's row count."""
    s = np.arange(-3000, 3001, dtype=np.float64)
    grid = [s / c for c in range(1, 67)]                                 # a read that clustering accepts has <= 66 rows
    rng = np.random.default_rng(3)
    big_s = np.round(np.sign(rng.standard_normal(200_000)) * 2.0 ** rng.uniform(0, 47, 200_000))
    big_c = np.floor(2.0 ** rng.uniform(0, np.log2(65534), 200_000))
    grid.append(big_s / big_c)
    grid.append(np.array([1.0, -1.0, 7.0, 1.0, 3.0]) / np.array([20000, 20000, 65534, 65534, 19999]))   # below 1e-4
    _check(np.concatenate(grid))


def test_edges():
    v = [0.0, -0.0, 5e-324, -5e-324, 2.2250738585072014e-308, 2.225073858507201e-308, 1.7976931348623157e308,
         -1.7976931348623157e308, 1e-4, 9.999999999999999e-05, 0.00010000000000000002, 1e16, 9999999999999998.0, 1.0000000000000002e16,
         1e15, 123456789012345.6, 0.1, 0.2, 0.30000000000000004, 1 / 3, 2 / 3, 464.6666666666667, 2066.6666666666665,
         6.666666666666667e-05, 9007199254740993.0, 1e23, 9.999999999999999e22, 5e-5, 1.5]
    v += [10.0 ** k for k in range(-5, 18)] + [float("1e%d" % k) for k in range(-5, 18)]
    v += [np.nextafter(10.0 ** k, 0) for k in range(-5, 18)] + [np.nextafter(10.0 ** k, np.inf) for k in range(-5, 18)]
    v += [2.0 ** k for k in range(-1074, 1024)] + [-(2.0 ** k) for k in range(-1074, 1024, 7)]
    v += [np.nextafter(2.0 ** k, 0) for k in range(-1022, 1024)]
    _check(np.array(v, dtype=np.float64))
