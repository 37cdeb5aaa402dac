"""ctypes wrapper of oracle/cpu_ref.c (C restatement of the reference's CPU algorithms; kind = "port").
TEST INFRASTRUCTURE + CPU BASELINE ONLY -- see the header of cpu_ref.c.  PARITY UNPINNED vs the Rust crates."""
from __future__ import annotations

import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile
from ctypes import c_int, c_size_t, c_uint64, c_void_p
from pathlib import Path

_DIR = Path(__file__).resolve().parent
_LIB = _DIR / "libvdf_cpu_ref.so"
_lib = None
_tmp_lib = None


def _host_signature() -> str:
    """CPU model + ISA flags of this machine: the library is compiled with -march=native, so a copy built on another
    host (the build container vs the GPU box) is rebuilt before it is loaded."""
    import hashlib
    model, flags = "", ""
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name") and not model:
                model = line.split(":", 1)[1].strip()
            elif line.startswith("flags") and not flags:
                flags = line.split(":", 1)[1].strip()
    except OSError:
        pass
    return model + " " + hashlib.sha1(flags.encode()).hexdigest()[:12]


def _make(out: Path) -> None:
    try:
        subprocess.run(["make", "-s", "-B", "-C", str(_DIR), f"OUT={out}"], check=True)
    except (subprocess.CalledProcessError, OSError):
        subprocess.run(["make", "-s", "-B", "-C", str(_DIR), f"OUT={out}", "ARCH=x86-64-v3"], check=True)


def build() -> Path:
    """Path of a library compiled for this host: the one beside the source, rebuilt there when it is stale, or -- when
    the tree is read-only -- a copy compiled into a temporary directory that is removed when the process exits."""
    global _tmp_lib
    sig_file = _DIR / "libvdf_cpu_ref.host"
    sig = _host_signature()
    stale = (not _LIB.exists() or _LIB.stat().st_mtime < (_DIR / "cpu_ref.c").stat().st_mtime
             or not sig_file.exists() or sig_file.read_text() != sig)
    if not stale:
        return _LIB
    if os.access(_DIR, os.W_OK):
        _make(_LIB)
        sig_file.write_text(sig)
        return _LIB
    if _tmp_lib is None:
        tmp = tempfile.mkdtemp(prefix="vdf_cpu_ref-")
        atexit.register(shutil.rmtree, tmp, True)
        _make(Path(tmp) / _LIB.name)
        _tmp_lib = Path(tmp) / _LIB.name
    return _tmp_lib


def load() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(str(build()))
    return _lib


def ncores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def _p(b):
    if b is None:
        return c_void_p(None)
    if isinstance(b, (bytes,)):
        return ctypes.cast(ctypes.c_char_p(b), c_void_p)
    if isinstance(b, bytearray):
        return ctypes.cast((ctypes.c_char * len(b)).from_buffer(b), c_void_p)
    if hasattr(b, "ctypes"):
        return c_void_p(b.ctypes.data)
    raise TypeError(type(b))


def msm(curve: int, affine72: bytes, scalars: bytes, is_mont: bool = True, nthreads: int = 0) -> bytes:
    out = bytearray(96)
    n = len(scalars) // 32
    load().ref_msm(c_int(curve), _p(affine72), c_size_t(n), _p(scalars), c_int(1 if is_mont else 0),
                   c_int(nthreads or ncores()), _p(out))
    return bytes(out)


def progression(curve: int, k0: int, d: int, n: int, nthreads: int = 0) -> bytes:
    out = bytearray(72 * n)
    load().ref_progression_mt(c_int(curve), _p(k0.to_bytes(32, "little")), _p(d.to_bytes(32, "little")), c_size_t(n),
                              c_int(nthreads or ncores()), _p(out))
    return bytes(out)


def minroot_check(field: int, results: bytes, originals: bytes, t, nthreads: int = 0) -> bytes:
    n = len(results) // 96
    ok = bytearray(n)
    if isinstance(t, int):
        load().ref_minroot_check(c_int(field), _p(results), _p(originals), c_void_p(None), c_uint64(t), c_size_t(n),
                                 c_int(nthreads or ncores()), _p(ok))
    else:
        import struct
        tb = struct.pack("<%dQ" % n, *t)
        load().ref_minroot_check(c_int(field), _p(results), _p(originals), _p(tb), c_uint64(0), c_size_t(n),
                                 c_int(nthreads or ncores()), _p(ok))
    return bytes(ok)


def multiply_vec(field: int, cons: int, nvars: int, io: int, coo, W: bytes, u: bytes, X: bytes, nthreads: int = 3) -> bytes:
    """coo = [(rows_u64_bytes, cols_u64_bytes, vals_bytes, nnz)] * 3 (oracle.pasta.shape_to_coo_bytes)."""
    out = bytearray(3 * cons * 32)
    args = []
    for rows, cols, vals, nnz in coo:
        args += [_p(rows), _p(cols), _p(vals), c_size_t(nnz)]
    load().ref_multiply_vec(c_int(field), c_size_t(cons), c_size_t(nvars), c_size_t(io), *args, _p(W), _p(u), _p(X),
                            c_int(nthreads), _p(out))
    return bytes(out)


def cross_term(field: int, cons: int, abc1: bytes, abc2: bytes, u1: bytes) -> bytes:
    out = bytearray(cons * 32)
    load().ref_cross_term(c_int(field), c_size_t(cons), _p(abc1), _p(abc2), _p(u1), _p(out))
    return bytes(out)


def fold(field: int, a: bytes, b: bytes, r: bytes) -> bytes:
    out = bytearray(a)
    load().ref_fold(c_int(field), _p(out), _p(b), c_size_t(len(a) // 32), _p(r))
    return bytes(out)


def field_mul(field: int, a: bytes, b: bytes) -> bytes:
    out = bytearray(len(a))
    load().ref_field_mul(c_int(field), _p(a), _p(b), c_size_t(len(a) // 32), _p(out))
    return bytes(out)
