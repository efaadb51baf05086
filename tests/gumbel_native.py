"""Builds and loads tests/native/gumbel_check.cpp (the host compile of the Gumbel draw of csrc/rng.cuh) into a temporary
directory, so that a read-only checkout can run the tests."""
import ctypes as C
import os
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "native", "gumbel_check.cpp")
_lib = None


def gumbel_lib():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="gumbel_check_"), "libgumbelcheck.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", SRC, "-o", out])
        lib = C.CDLL(out)
        for name in ("gc_gumbel", "gc_uniform"):
            f = getattr(lib, name)
            f.restype = C.c_double
            f.argtypes = [C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32]
        _lib = lib
    return _lib


def host_draws(seed: int, uid: int, search_index: int, ply: int, A: int):
    lib = gumbel_lib()
    lo, hi = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    return [lib.gc_gumbel(lo, hi, uid, search_index, ply, a) for a in range(A)]
