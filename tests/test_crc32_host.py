"""CPU tests of the CRC-32 that checks BGZF blocks on the device (fslr_b200/csrc/crc32.cuh), host build against zlib: the
sequential update, the 32-lane split of k_bgzf_crc with its shift-and-XOR combine, and the shift constants."""
import ctypes
import os
import subprocess
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "tests", "_build")
LENGTHS = [0, 1, 7, 8, 9, 15, 16, 17, 2047, 2048, 2049, 4095, 4096, 63488, 65535, 65536]


def _lib():
    os.makedirs(BUILD, exist_ok=True)
    so = os.path.join(BUILD, "libhost_crc32.so")
    deps = [os.path.join(ROOT, "tests", "host_crc32_harness.cpp"), os.path.join(ROOT, "fslr_b200", "csrc", "crc32.cuh")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", "-o", so, deps[0]])
    lib = ctypes.CDLL(so)
    for f in (lib.host_crc32, lib.host_crc32_lanes, lib.host_multmodp, lib.host_shift):
        f.restype = ctypes.c_uint32
    lib.host_crc32.argtypes = [ctypes.c_void_p, ctypes.c_longlong]
    lib.host_crc32_lanes.argtypes = [ctypes.c_void_p, ctypes.c_int]
    lib.host_multmodp.argtypes = [ctypes.c_uint32, ctypes.c_uint32]
    lib.host_shift.argtypes = [ctypes.c_int]
    return lib


def _cases():
    """(buffer, start, length): every listed length and 200 random ones up to 65536, at every start alignment mod 16
    (a BGZF block's inflated bytes start wherever the ISIZEs before it put them)."""
    rng = np.random.default_rng(11)
    buf = rng.integers(0, 256, 65536 + 64, dtype=np.uint8)
    lengths = LENGTHS + [int(x) for x in rng.integers(0, 65537, 200)]
    for i, n in enumerate(lengths):
        yield buf, i % 16, n


def test_sequential_crc_equals_zlib():
    lib = _lib()
    for buf, a, n in _cases():
        assert lib.host_crc32(buf.ctypes.data + a, n) == zlib.crc32(buf[a:a + n].tobytes()), (a, n)
    text = b"ACGT" * 20000                                                    # low-entropy bytes too
    assert lib.host_crc32(text, len(text)) == zlib.crc32(text)


def test_lane_split_equals_zlib():
    lib = _lib()
    for buf, a, n in _cases():
        assert lib.host_crc32_lanes(buf.ctypes.data + a, n) == zlib.crc32(buf[a:a + n].tobytes()), (a, n)
    for a in range(16):                                                      # every alignment at the sizes a lane boundary
        for n in (2047, 2048, 2049, 65536):                                   # or the first lane sits on
            buf = np.random.default_rng(a * 100000 + n).integers(0, 256, n + 16, dtype=np.uint8)
            assert lib.host_crc32_lanes(buf.ctypes.data + a, n) == zlib.crc32(buf[a:a + n].tobytes()), (a, n)


def test_multmodp_by_x0_is_the_identity():
    lib = _lib()
    for v in [0, 1, 0xFFFFFFFF, 0x80000000] + [int(x) for x in np.random.default_rng(3).integers(0, 1 << 32, 100)]:
        assert lib.host_multmodp(1 << 31, v) == v


def test_shift_constants_combine_like_zlib():
    """zlib's crc32_combine: crc(A + B) = multmodp(x^(8 len(B)), crc(A)) ^ crc(B); the kernel's shift[j] is that
    constant for len(B) = j * 2048."""
    lib = _lib()
    rng = np.random.default_rng(5)
    assert lib.host_shift(0) == 1 << 31
    for j in range(32):
        a = rng.integers(0, 256, int(rng.integers(1, 3000)), dtype=np.uint8).tobytes()
        b = rng.integers(0, 256, j * 2048, dtype=np.uint8).tobytes()
        assert lib.host_multmodp(lib.host_shift(j), zlib.crc32(a)) ^ zlib.crc32(b) == zlib.crc32(a + b), j
