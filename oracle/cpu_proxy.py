"""ctypes wrapper over oracle/cpu_proxy.cc — the "fused-cxx-proxy" CPU arm of bench.py.

BENCH / TEST INFRASTRUCTURE ONLY (see oracle/__init__.py): imported by bench.py's `cpu_baseline` and
`--impl reference` legs and by tests/test_cpu_proxy.py, never by anything under gandiva_b200/.

The library is compiled on first use ON THE MACHINE THAT RUNS IT with `g++ -O3 -march=native`
(`oracle/_proxy/libgdv_cpu_proxy_<cpu-flags-hash>.so`, git-ignored): a `.so` built in the GPU-less
container travels to the GPU box, whose host CPU may have a different instruction set, so the file
name carries a hash of /proc/cpuinfo's flags and a mismatch triggers a one-second rebuild.  The build step
(gandiva_b200/build.py) writes the in-tree file; a rebuild at run time goes to the temporary directory
(`gdv_cpu_proxy_<uid>/`), so that the benchmark also runs from a read-only tree.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_DIR = os.path.join(_HERE, "_proxy")
CXXFLAGS = ["-O3", "-march=native", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-pthread"]


def _cpu_key() -> str:
    flags = ""
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("flags"):
                flags = ln
                break
    except OSError:
        pass
    src = open(os.path.join(_HERE, "cpu_proxy.cc"), "rb").read() + open(os.path.join(_HERE, "lineitem.h"), "rb").read()
    return hashlib.sha1(flags.encode() + src).hexdigest()[:12]


def build(directory: str = _DIR) -> str:
    path = os.path.join(directory, "libgdv_cpu_proxy_%s.so" % _cpu_key())
    if not os.path.exists(path):
        os.makedirs(directory, exist_ok=True)
        tmp = path + ".tmp%d" % os.getpid()
        subprocess.check_call(["g++"] + CXXFLAGS + [os.path.join(_HERE, "cpu_proxy.cc"), "-o", tmp])
        os.replace(tmp, path)
    return path


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        path = os.path.join(_DIR, "libgdv_cpu_proxy_%s.so" % _cpu_key())
        if not os.path.exists(path):   # a CPU the in-tree build did not see: the tree may be read-only
            path = build(os.path.join(tempfile.gettempdir(), "gdv_cpu_proxy_%d" % os.getuid()))
        L = C.CDLL(path)
        vp, i64 = C.c_void_p, C.c_int64
        L.proxy_threads.restype = C.c_int
        L.proxy_threads.argtypes = [C.c_int]
        L.proxy_simd.restype = C.c_int
        L.proxy_alloc.restype = vp
        L.proxy_alloc.argtypes = [C.c_size_t]
        L.proxy_free.argtypes = [vp]
        L.proxy_generate.argtypes = [C.c_int, C.c_uint64, i64, i64, vp, vp, C.c_int, C.c_int]
        L.proxy_copy_rows.argtypes = [vp, vp, i64, C.c_int, C.c_int]
        L.proxy_q6_filter.restype = i64
        L.proxy_q6_filter.argtypes = [vp, vp, vp, vp, vp, vp, i64, vp, vp, C.c_int]
        L.proxy_add_i32.argtypes = [vp, vp, vp, vp, i64, vp, vp, C.c_int]
        L.proxy_add_i32_inline.argtypes = [vp, vp, vp, vp, i64, vp, vp]
        L.proxy_comment_filter.restype = i64
        L.proxy_comment_filter.argtypes = [vp, vp, vp, i64, vp, vp, C.c_int]
        L.proxy_q1_project.argtypes = [C.POINTER(vp), C.POINTER(vp), i64, C.POINTER(vp), C.POINTER(vp), C.c_int]
        _lib = L
    return _lib


def threads(want: int = 0) -> int:
    """Size of the pinned pool (fixed by the first call in the process)."""
    return int(lib().proxy_threads(want))


def simd() -> str:
    return "avx512" if lib().proxy_simd() == 512 else "compiler auto-vectorisation"


class Buf:
    """Page-aligned host memory that is first touched by the pool's threads, as a numpy view."""

    def __init__(self, count: int, dtype):
        self.dtype = np.dtype(dtype)
        self.count = count
        self.nbytes = max(count * self.dtype.itemsize, 64)
        self.ptr = lib().proxy_alloc(self.nbytes)
        if not self.ptr:
            raise MemoryError("proxy_alloc(%d)" % self.nbytes)
        self.array = np.ctypeslib.as_array(C.cast(self.ptr, C.POINTER(C.c_uint8)), shape=(self.nbytes,))[
            : count * self.dtype.itemsize].view(self.dtype)

    def free(self):
        if self.ptr:
            self.array = None
            lib().proxy_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


_KIND_DTYPE = {0: np.int32, 1: np.float64, 2: np.float64, 3: np.int64, 7: np.float64, 8: np.float64, 9: np.int32,
               10: np.int32}


def generate(kind: int, seed: int, first_row: int, n: int, null_permille: int = 0):
    """A lineitem column (oracle/lineitem.h) filled by the pool: returns (values Buf, validity Buf | None)."""
    if kind in (4, 5, 6):
        vals = Buf(2 * n, np.uint64)
    else:
        vals = Buf(n, _KIND_DTYPE.get(kind, np.int32))
    vld = Buf((n + 7) // 8 + 8, np.uint8) if null_permille > 0 else None
    lib().proxy_generate(kind, seed, first_row, n, vals.ptr, vld.ptr if vld else None, null_permille, 0)
    return vals, vld


def _p(x):
    if x is None:
        return None
    if isinstance(x, Buf):
        return x.ptr
    return x.ctypes.data


def q6_filter(ship, disc, qty, v_ship, v_disc, v_qty, n: int, out, bits) -> int:
    return int(lib().proxy_q6_filter(_p(ship), _p(disc), _p(qty), _p(v_ship), _p(v_disc), _p(v_qty), n, _p(out),
                                     _p(bits), 0))


def add_i32(a, b, va, vb, n: int, out, vout) -> None:
    lib().proxy_add_i32(_p(a), _p(b), _p(va), _p(vb), n, _p(out), _p(vout), 0)


def add_i32_inline(a, b, va, vb, n: int, out, vout) -> None:
    """On the calling thread only (one batch, one thread: how the reference evaluates a RecordBatch)."""
    lib().proxy_add_i32_inline(_p(a), _p(b), _p(va), _p(vb), n, _p(out), _p(vout))


def comment_filter(offsets, data, validity, n: int, out, bits) -> int:
    return int(lib().proxy_comment_filter(_p(offsets), _p(data), _p(validity), n, _p(out), _p(bits), 0))


def q1_project(ins, vins, n: int, outs, vouts) -> None:
    A = C.c_void_p * 8
    lib().proxy_q1_project(A(*[_p(x) for x in ins]), A(*[_p(x) for x in vins]), n, A(*[_p(x) for x in outs]),
                           A(*[_p(x) for x in vouts]), 0)
