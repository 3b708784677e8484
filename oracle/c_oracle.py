"""TEST INFRASTRUCTURE ONLY -- ctypes loader for the plain-C oracle (oracle/copy_rects_ref.c).

The oracle consumes the product's tsb_rect_t descriptors with HOST pointers, so a test can hand
the same descriptors to the CUDA kernel and to this library and compare bytes.
"""

from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "_build", "liboracle_copy_rects.so")

_lib = None


def _writable_dir(path: str) -> bool:
    try:
        os.makedirs(path, exist_ok=True)
    except OSError:
        return False
    return os.access(path, os.W_OK)


def build(force: bool = False) -> str:
    """Compile the oracle into oracle/_build when it is missing or older than its sources; returns the
    library's path.  A checkout that cannot be written (bench.py may run from a read-only tree) gets
    the rebuild in a temporary directory, removed at exit."""
    src = os.path.join(HERE, "copy_rects_ref.c")
    hdr = os.path.join(os.path.dirname(HERE), "include", "tstore_b200.h")
    stale = (not os.path.exists(LIB)) or os.path.getmtime(LIB) < max(os.path.getmtime(src), os.path.getmtime(hdr))
    if not (force or stale):
        return LIB
    out = LIB
    if not _writable_dir(os.path.dirname(LIB)):
        tmp_dir = tempfile.mkdtemp(prefix="tsb_oracle_")
        atexit.register(shutil.rmtree, tmp_dir, True)
        out = os.path.join(tmp_dir, os.path.basename(LIB))
    cmd = ["gcc", "-O2", "-fPIC", "-shared", "-pthread", "-std=gnu11", "-I", os.path.dirname(hdr), "-o", out + ".tmp", src]
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError(f"oracle build failed:\n{proc.stdout}\n{proc.stderr}")
    os.replace(out + ".tmp", out)
    return out


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        h = C.CDLL(build())
        h.oracle_copy_rects.restype = C.c_int
        h.oracle_copy_rects.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_int]
        h.oracle_copy_rects_pinned.restype = C.c_int
        h.oracle_copy_rects_pinned.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_int]
        h.oracle_convert.restype = C.c_int
        h.oracle_convert.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint64, C.c_int]
        h.oracle_replay_plan.restype = C.c_int
        h.oracle_replay_plan.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_uint32, C.c_int]
        _lib = h
    return _lib


def copy_rects(rects, n: int, nan_mode: int = 0, nthreads: int = 1, pin: bool = False) -> None:
    """rects: ctypes array of tsb_rect_t (torchstore_b200._native.Rect) with host pointers.
    pin=True binds worker t to the t-th allowed core (stable NUMA placement for bench.py's baseline)."""
    fn = lib().oracle_copy_rects_pinned if pin else lib().oracle_copy_rects
    st = fn(C.cast(rects, C.c_void_p), n, nan_mode, nthreads)
    if st != 0:
        raise RuntimeError(f"oracle_copy_rects failed with {st}")


def convert(src_ptr: int, src_code: int, dst_ptr: int, dst_code: int, n: int, nan_mode: int = 0) -> None:
    st = lib().oracle_convert(C.c_void_p(src_ptr), src_code, C.c_void_p(dst_ptr), dst_code, n, nan_mode)
    if st != 0:
        raise RuntimeError(f"oracle_convert failed with {st}")


def replay_plan(rect_table, tiles, tile_units: int, nan_mode: int = 0) -> None:
    """Replay tables from tsb_plan_compile_host (numpy arrays) on host memory."""
    n_rects = rect_table.size // 192
    st = lib().oracle_replay_plan(C.c_void_p(rect_table.ctypes.data), n_rects, C.c_void_p(tiles.ctypes.data),
                                  tiles.shape[0], tile_units, nan_mode)
    if st != 0:
        raise RuntimeError(f"oracle_replay_plan failed with {st}")
