"""CPU: the inner-product argument's device functors (sumcheck.cuh IpaExpandFn, IpaFoldFn) run by a CPU loop
(tests/emul/emul_ipa.cpp) against tests/ipa_ref.py, round by round: the commitment scalars SL / SR over G[0, n]
including slot n, the folded a and b, coef_j after every round and coef_ell = s.  And the argument errors of the three
IPA entry points, which come back before any device work, with or without a GPU."""
import ctypes
import random
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import pasta as O
from tests import ipa_ref as IR
from tests.util import aligned, ptr
from vdf_b200 import _lib

ROOT = Path(__file__).resolve().parent.parent
SZ = ctypes.c_size_t
ERR_ARG = -1


@pytest.fixture(scope="module")
def emul_ipa(tmp_path_factory):
    src = ROOT / "tests" / "emul" / "emul_ipa.cpp"
    lib = tmp_path_factory.mktemp("emul_ipa") / "libvdf_emul_ipa.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", str(lib), str(src)],
                   check=True)
    return ctypes.CDLL(str(lib))


def _buf(vals, m):
    return aligned(O.fes_to_bytes(vals, m) or bytes(32))


def _vals(arr, count, m):
    return O.fes_from_bytes(arr.tobytes()[:32 * count], m)


@pytest.mark.parametrize("fid", [O.FIELD_FP, O.FIELD_FQ])
@pytest.mark.parametrize("ell", [1, 2, 3, 7])
def test_expand_and_fold_match_reference(emul_ipa, fid, ell):
    m = O.MODULUS[fid]
    py = random.Random(ell * 10 + fid)
    n = 1 << ell
    a = [py.randrange(m) for _ in range(n)]
    b = [py.randrange(m) for _ in range(n)]
    a[0] = 0
    b[-1] = m - 1
    u_scale = py.randrange(1, m)
    rs = [py.randrange(1, m) for _ in range(ell)]
    rs[-1] = 1 if ell > 1 else m - 1
    want_coef = IR.coef_tables(rs, m)
    # the device state: a and b halved in place, coef ping-ponging between two n-entry buffers
    da, db = _buf(a, m), _buf(b, m)
    coef = [aligned(bytes(32 * n)), aligned(bytes(32 * n))]
    coef[0][:32] = np.frombuffer(O.fe_to_bytes(1, m), np.uint8)
    SL, SR = aligned(bytes(32 * (n + 1))), aligned(bytes(32 * (n + 1)))
    ra, rb = list(a), list(b)
    for j, r in enumerate(rs):
        mm = n >> j
        h = mm // 2
        cL, cR = IR.inner(ra[:h], rb[h:], m), IR.inner(ra[h:], rb[:h], m)
        wantL, wantR = IR.expand(ra, want_coef[j], n, cL, cR, u_scale, m)
        c2, us = _buf([cL, cR], m), _buf([u_scale], m)
        emul_ipa.emul_ipa_expand(fid, ptr(da), ptr(coef[j & 1]), ptr(c2), ptr(us), ctypes.c_uint32(ell - j), SZ(n),
                                 ptr(SL), ptr(SR))
        assert _vals(SL, n + 1, m) == wantL, j
        assert _vals(SR, n + 1, m) == wantR, j
        # slot n carries the c U term; the scalars of G[0, n) are non-zero on one side of every pair only
        assert wantL[n] == cL * u_scale % m and wantR[n] == cR * u_scale % m
        rb_, ri_ = _buf([r], m), _buf([pow(r, -1, m)], m)
        emul_ipa.emul_ipa_fold(fid, ptr(da), ptr(db), SZ(h), ptr(coef[j & 1]), ptr(coef[(j & 1) ^ 1]), SZ(1 << j),
                               ptr(rb_), ptr(ri_))
        ra, rb = IR.fold(ra, rb, r, m)
        assert _vals(da, h, m) == ra and _vals(db, h, m) == rb, j
        assert _vals(coef[(j & 1) ^ 1], 2 << j, m) == want_coef[j + 1], j
    assert _vals(coef[ell & 1], n, m) == IR.s_table(rs, m)
    # h = 0 only doubles the table: the s table of vdfgpu_ipa_gens_hat
    t = [aligned(bytes(32 * n)), aligned(bytes(32 * n))]
    t[0][:32] = np.frombuffer(O.fe_to_bytes(1, m), np.uint8)
    for j, r in enumerate(rs):
        emul_ipa.emul_ipa_fold(fid, None, None, SZ(0), ptr(t[j & 1]), ptr(t[(j & 1) ^ 1]), SZ(1 << j),
                               ptr(_buf([r], m)), ptr(_buf([pow(r, -1, m)], m)))
    assert _vals(t[ell & 1], n, m) == IR.s_table(rs, m)


def test_s_table_is_novas_recurrence():
    """nova's s: s[0] = prod r^-1, s[i] = s[i - 2^pos] r^2_{ell-1-pos} with 2^pos the highest power of two <= i"""
    m = O.Q
    py = random.Random(5)
    rs = [py.randrange(1, m) for _ in range(5)]
    ell = len(rs)
    s = [1]
    for r in rs:
        s[0] = s[0] * pow(r, -1, m) % m
    for i in range(1, 1 << ell):
        pos = i.bit_length() - 1
        s.append(s[i - (1 << pos)] * rs[ell - 1 - pos] ** 2 % m)
    assert s == IR.s_table(rs, m) == IR.coef_tables(rs, m)[-1]


# Zeroed host memory behind every pointer argument.  Without a GPU no generator set can be built, so the non-null
# handle is this buffer too: it relies on struct vdfgpu_gens (vdf_b200/csrc/ctx.cuh) lying within its first bytes, so
# that the set reads as 0 points and every ell is "too few points".  The null checks come before any read of it.
_mem = ctypes.create_string_buffer(1 << 12)
_cb = _lib.IPA_ROUND_FN(lambda *a: 0)


def _calls():
    cb = ctypes.cast(_cb, ctypes.c_void_p)
    g = ctypes.addressof(_mem)
    return {
        "prove: null gens": lambda lib: lib.vdfgpu_ipa_prove(None, _mem, _mem, 1, _mem, cb, None, _mem),
        "prove: null a": lambda lib: lib.vdfgpu_ipa_prove(g, None, _mem, 1, _mem, cb, None, _mem),
        "prove: null b": lambda lib: lib.vdfgpu_ipa_prove(g, _mem, None, 1, _mem, cb, None, _mem),
        "prove: null u_scale": lambda lib: lib.vdfgpu_ipa_prove(g, _mem, _mem, 1, None, cb, None, _mem),
        "prove: null callback": lambda lib: lib.vdfgpu_ipa_prove(g, _mem, _mem, 1, _mem, None, None, _mem),
        "prove: null a_hat": lambda lib: lib.vdfgpu_ipa_prove(g, _mem, _mem, 1, _mem, cb, None, None),
        "prove: host form ell > 30": lambda lib: lib.vdfgpu_ipa_prove(g, _mem, _mem, 31, _mem, cb, None, _mem),
        "prove: too few points": lambda lib: lib.vdfgpu_ipa_prove(g, _mem, _mem, 0, _mem, cb, None, _mem),
        "prove_dev: null gens": lambda lib: lib.vdfgpu_ipa_prove_dev(None, _mem, _mem, 1, _mem, cb, None, _mem),
        "prove_dev: null callback": lambda lib: lib.vdfgpu_ipa_prove_dev(g, _mem, _mem, 1, _mem, None, None, _mem),
        "prove_dev: null a_hat": lambda lib: lib.vdfgpu_ipa_prove_dev(g, _mem, _mem, 1, _mem, cb, None, None),
        "prove_dev: ell 63": lambda lib: lib.vdfgpu_ipa_prove_dev(g, _mem, _mem, 63, _mem, cb, None, _mem),
        "gens_hat: null gens": lambda lib: lib.vdfgpu_ipa_gens_hat(None, _mem, 1, _mem),
        "gens_hat: null r": lambda lib: lib.vdfgpu_ipa_gens_hat(g, None, 1, _mem),
        "gens_hat: null output": lambda lib: lib.vdfgpu_ipa_gens_hat(g, _mem, 1, None),
        "gens_hat: too few points": lambda lib: lib.vdfgpu_ipa_gens_hat(g, _mem, 0, _mem),
    }


@pytest.mark.parametrize("case", sorted(_calls()))
def test_argument_errors_launch_nothing(case):
    lib = _lib.load()
    launches = lib.vdfgpu_launch_count()
    assert _calls()[case](lib) == ERR_ARG, lib.vdfgpu_last_error()
    assert lib.vdfgpu_last_error().decode().startswith("ipa_")
    assert lib.vdfgpu_launch_count() == launches
