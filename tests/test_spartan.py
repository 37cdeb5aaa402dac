"""CPU: the Spartan prover's device functors (r1cs.cuh PaddedLayout, OuterTablesFn, PaddedScatterFn; sumcheck.cuh
MultiDot, IpaJoinFn) run by a CPU loop (tests/emul/emul_spartan.cpp) against tests/spartan_ref.py; spartan_ref itself
against the two-phase semantics and the inner-product argument it ends in; and the argument errors of
vdfgpu_running_spartan_prove and vdfgpu_r1cs_evaluate, which come back before any device work, with or without a GPU."""
import ctypes
import random
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import pasta as O
from tests import ipa_ref as IR
from tests import shape_gen as S
from tests import spartan_ref as SR
from tests.util import aligned, ptr
from vdf_b200 import _lib
from vdf_b200 import spartan as SP

ROOT = Path(__file__).resolve().parent.parent
SZ, U32 = ctypes.c_size_t, ctypes.c_uint32
ERR_ARG = -1
FIDS = [O.FIELD_FP, O.FIELD_FQ]


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    src = ROOT / "tests" / "emul" / "emul_spartan.cpp"
    lib = tmp_path_factory.mktemp("emul_spartan") / "libvdf_emul_spartan.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", str(lib), str(src)],
                   check=True)
    lib = ctypes.CDLL(str(lib))
    lib.emul_padded_layout.restype = ctypes.c_uint64
    return lib


def _buf(vals, m):
    return aligned(O.fes_to_bytes(vals, m) or bytes(32))


def _vals(arr, count, m):
    return O.fes_from_bytes(arr.tobytes()[:32 * count], m)


def _csr(shape):
    """the library's stacked CSR: rows A 0..cons-1, then B, then C; entries in COO order within a row"""
    rows = [[] for _ in range(3 * shape.num_cons)]
    for k, M in enumerate((shape.A, shape.B, shape.C)):
        for r, c, v in M:
            rows[k * shape.num_cons + r].append((c, v))
    row_ptr = np.zeros(len(rows) + 1, np.uint32)
    row_ptr[1:] = np.cumsum([len(r) for r in rows])
    col = np.array([c for r in rows for c, _ in r] or [0], np.uint32)
    val = _buf([v for r in rows for _, v in r], shape.m)
    return row_ptr, col, val


# (cons, vars, io): vars < m, vars = m, cons = m with io = 0, both below m with io = 7
SHAPES = [(45, 40, 7), (30, 64, 2), (64, 20, 0), (33, 50, 7)]


@pytest.mark.parametrize("cons,vars_,io", SHAPES + [(1, 1, 0), (1, 1, 1), (5, 3, 4), (100, 2, 200)])
def test_padded_layout(emul, cons, vars_, io):
    shape = O.R1CSShape(O.Q, cons, vars_, io, [], [], [])
    m = SR.padded_size(shape)
    fits = ctypes.c_int()
    cols = np.zeros(vars_ + 1 + io, np.uint64)
    src = np.zeros(2 * m, np.int64)
    assert emul.emul_padded_layout(U32(cons), U32(vars_), U32(io), ctypes.byref(fits), ptr(cols), ptr(src)) == m
    assert bool(fits.value) == (1 + io <= m)
    m_py, col = SP.padded_layout(cons, vars_, io)
    assert m_py == m
    want = [c if c < vars_ else c + m - vars_ for c in range(vars_ + 1 + io)]
    assert list(cols) == want == [col(c) for c in range(vars_ + 1 + io)]
    if fits.value:   # source() inverts col() and marks every other slot of [0, 2m) as padding
        inv = {p: c for c, p in enumerate(want)}
        assert list(src) == [inv.get(j, -1) for j in range(2 * m)]


@pytest.mark.parametrize("fid", FIDS)
@pytest.mark.parametrize("cons,vars_,io", SHAPES)
def test_outer_tables(emul, fid, cons, vars_, io):
    """Az, Bz, Cz and D = u Cz + E over the m padded rows, u != 1, E != 0, zero rows past cons"""
    shape = S.general_shape(fid, cons, vars_, io)
    p = shape.m
    W, _, u, X = S.relaxed_instance(shape, seed=cons)
    E = S.random_vec(random.Random(cons), p, cons)
    m = SR.padded_size(shape)
    row_ptr, col, val = _csr(shape)
    out = aligned(bytes(4 * 32 * m))
    emul.emul_outer_tables(fid, ptr(row_ptr), ptr(col), ptr(val), U32(cons), U32(vars_), U32(io), ptr(_buf(W, p)),
                           ptr(_buf([u] + X, p)), ptr(_buf(E + [0] * (m - cons), p)), SZ(m), ptr(out))
    got = _vals(out, 4 * m, p)
    Az, Bz, Cz = (v + [0] * (m - cons) for v in shape.multiply_vec(shape.z_of(W, u, X)))
    D = [(u * c + e) % p for c, e in zip(Cz, E)] + [0] * (m - cons)
    assert got[:m] == Az and got[m:2 * m] == Bz and got[2 * m:3 * m] == Cz and got[3 * m:] == D
    assert u != 1 and any(E)


@pytest.mark.parametrize("fid", FIDS)
@pytest.mark.parametrize("cons,vars_,io", SHAPES)
def test_padded_scatter(emul, fid, cons, vars_, io):
    """M and z written at the padded columns of a 2m-entry table, zero elsewhere"""
    shape = S.general_shape(fid, cons, vars_, io)
    p = shape.m
    py = random.Random(vars_)
    W, u, X = S.random_vec(py, p, vars_), py.randrange(2, p), S.random_vec(py, p, io)
    eq_rows, r_abc = S.random_vec(py, p, cons), [py.randrange(p) for _ in range(3)]
    M = shape.bind_rows(eq_rows, r_abc)
    m = SR.padded_size(shape)
    Mp, zp = aligned(bytes(64 * m)), aligned(bytes(64 * m))
    emul.emul_padded_scatter(fid, U32(cons), U32(vars_), U32(io), ptr(_buf(M, p)), ptr(_buf(W, p)),
                             ptr(_buf([u] + X, p)), ptr(Mp), ptr(zp))
    want_M = [0] * (2 * m)
    for Mat, rm in zip(SR.padded_entries(shape), r_abc):
        for r, c, v in Mat:
            want_M[c] = (want_M[c] + rm * v % p * eq_rows[r]) % p
    assert _vals(Mp, 2 * m, p) == want_M
    assert _vals(zp, 2 * m, p) == SR.padded_z(shape, W, u, X)


@pytest.mark.parametrize("fid", FIDS)
def test_multi_dot_with_short_vectors(emul, fid):
    """three inner products in one pass, each vector with its own length below the table length: nothing past it read"""
    p = O.MODULUS[fid]
    py = random.Random(7 + fid)
    n = 64
    for lens in ((64, 64, 64), (45, 64, 1), (0, 33, 63)):
        vs = [S.random_vec(py, p, k) for k in lens]
        eqs = [O.eq_evals([py.randrange(p) for _ in range(6)], p) for _ in range(3)]
        bv = [_buf(v + [p - 1] * 4, p) for v in vs]   # entries past len are non-zero: they must not count
        be = [_buf(e, p) for e in eqs]
        vp = (ctypes.c_void_p * 3)(*[b.ctypes.data for b in bv])
        ep = (ctypes.c_void_p * 3)(*[b.ctypes.data for b in be])
        out = aligned(bytes(96))
        emul.emul_multi_dot3(fid, vp, ep, (SZ * 3)(*lens), SZ(n), ptr(out))
        assert _vals(out, 3, p) == [IR.inner(v, e, p) for v, e in zip(vs, eqs)], lens


@pytest.mark.parametrize("fid", FIDS)
def test_ipa_join(emul, fid):
    """a = E + rho W, b = eq(r_x) + rho eq(r_y'), in place too; <a, b> = eval_E + rho T + rho^2 eval_W"""
    p = O.MODULUS[fid]
    py = random.Random(11 + fid)
    n = 32
    E, W = S.random_vec(py, p, n), S.random_vec(py, p, n)
    rx, ry = [py.randrange(p) for _ in range(5)], [py.randrange(p) for _ in range(5)]
    eqx, eqy = O.eq_evals(rx, p), O.eq_evals(ry, p)
    rho = py.randrange(p)
    bE, bx = _buf(E, p), _buf(eqx, p)
    emul.emul_ipa_join(fid, ptr(bE), ptr(_buf(W, p)), ptr(bx), ptr(_buf(eqy, p)), ptr(_buf([rho], p)), SZ(n), ptr(bE),
                       ptr(bx))
    a, b = _vals(bE, n, p), _vals(bx, n, p)
    assert a == [(e + rho * w) % p for e, w in zip(E, W)]
    assert b == [(x + rho * y) % p for x, y in zip(eqx, eqy)]
    eval_E, eval_W = IR.inner(E, eqx, p), IR.inner(W, eqy, p)
    T = (IR.inner(E, eqy, p) + IR.inner(W, eqx, p)) % p
    assert IR.inner(a, b, p) == (eval_E + rho * T + rho * rho * eval_W) % p


def test_reference_prover_against_two_phase_semantics():
    """spartan_ref on a folded step instance (u != 1, E != 0): the rounds are the oracle's sum-checks over the padded
    tables, the verifier accepts, the opening verifies under comm_E + rho comm_W, and a wrong E entry is caught"""
    fid = O.FIELD_FQ
    cv = O.PALLAS
    p = O.Q
    shape, W1, X1, _ = O.make_step_instance(fid, 4, O.State(5, 6, 4))
    _, W2, X2, _ = O.make_step_instance(fid, 4, O.State(9, 1, 4))
    r = 1 + 2 ** 100
    T = shape.cross_term(W1, 1, X1, W2, X2)
    W, E, X, u = O.fold_vec(W1, W2, r, p), [r * t % p for t in T], O.fold_vec(X1, X2, r, p), (1 + r) % p
    assert shape.is_sat_relaxed(W, E, u, X) and any(E)
    m = SR.padded_size(shape)
    assert shape.num_vars < m and shape.num_cons < m
    py = random.Random(3)
    G = [cv.mul(py.randrange(1, cv.order), cv.gen) for _ in range(m + 1)]
    tau = [py.randrange(p) for _ in range(m.bit_length() - 1)]
    tr = SR.Transcript()
    pf = SR.prove(shape, W, E, u, X, tau, tr, cv, G)
    assert SR.transcript_consistent(pf, tr, p)
    assert SR.verify_claims(shape, u, X, tau, pf)
    # the outer rounds are the oracle's cubic sum-check over eq(tau), Az, Bz, u Cz + E padded to m rows
    Az, Bz, Cz = (v + [0] * (m - shape.num_cons) for v in shape.multiply_vec(shape.z_of(W, u, X)))
    D = [(u * c + e) % p for c, e in zip(Cz, E + [0] * (m - shape.num_cons))]
    evals, rx, _ = O.sumcheck_prove([O.eq_evals(tau, p), Az, Bz, D], p, lambda j, e: tr.sumcheck_round(j, tuple(e)) % p)
    assert [e for e, _ in pf.outer] == [tuple(e) for e in evals] and pf.r_x == rx
    # the opening: P = comm_E + rho comm_W + c U, b = eq(r_x) + rho eq(r_y')
    rys = pf.r_y[1:]
    comm = cv.add(cv.msm_naive(E + [0] * (m - len(E)), G[:m]), cv.mul(pf.rho, cv.msm_naive(W + [0] * (m - len(W)), G[:m])))
    b = [(x + pf.rho * y) % p for x, y in zip(O.eq_evals(rx, p), O.eq_evals(rys, p))]
    Ls, Rs, rs = [O.jac_from_bytes(cv, L) for L, _, _ in pf.ipa], [O.jac_from_bytes(cv, R) for _, R, _ in pf.ipa], \
        [r for _, _, r in pf.ipa]
    P = cv.add(comm, cv.mul(pf.c * pf.u_scale % p, G[m]))
    assert IR.verify(cv, G[:m], G[m], pf.u_scale, P, b, Ls, Rs, rs, pf.a_hat)
    assert SP.ipa_b_hat(fid, rs, [(1, rx), (pf.rho, rys)]) == IR.inner(b, IR.s_table(rs, p), p)
    # an unsatisfied instance: the prover still answers, the verifier rejects
    E_bad = list(E)
    E_bad[2] = (E_bad[2] + 1) % p
    assert not SR.verify_claims(shape, u, X, tau, SR.prove(shape, W, E_bad, u, X, tau, tr, cv, G))


# ---- argument errors, before any device work -------------------------------------------------------------------
# Without a GPU no shape, set or instance can be built, so the handles are host structures that mirror the leading
# fields of struct vdfgpu_r1cs, vdfgpu_gens and vdfgpu_running (vdf_b200/csrc/api_r1cs.cu, ctx.cuh): the checks read
# only those.
class _Shape(ctypes.Structure):
    _fields_ = [("field", ctypes.c_int), ("cons", ctypes.c_uint32), ("vars", ctypes.c_uint32), ("io", ctypes.c_uint32),
                ("rest", ctypes.c_uint8 * 256)]


class _Gens(ctypes.Structure):
    _fields_ = [("curve", ctypes.c_int), ("n", ctypes.c_size_t), ("rest", ctypes.c_uint8 * 256)]


class _Running(ctypes.Structure):
    _fields_ = [("shape", ctypes.c_void_p), ("gens", ctypes.c_void_p), ("rest", ctypes.c_uint8 * 512)]


_mem = ctypes.create_string_buffer(1 << 12)
_cbs = (_lib.ROUND_FN(lambda *a: 0), _lib.CLAIMS_FN(lambda *a: 0), _lib.IPA_ROUND_FN(lambda *a: 0))
_keep = []


def _running(cons, vars_, io, curve=O.CURVE_PALLAS, n=1 << 20):
    s = _Shape(O.FIELD_FQ, cons, vars_, io)
    g = _Gens(curve, n)
    f = _Running(ctypes.addressof(s), ctypes.addressof(g))
    _keep.extend((s, g, f))
    return ctypes.addressof(f), ctypes.addressof(g), ctypes.addressof(s)


def _calls():
    sc, cl, ipa = (ctypes.cast(c, ctypes.c_void_p) for c in _cbs)
    f, g, s = _running(100, 90, 2)
    prove = _lib.load().vdfgpu_running_spartan_prove
    return {
        "prove: null instance": lambda: prove(None, g, _mem, sc, cl, ipa, None, _mem),
        "prove: null set": lambda: prove(f, None, _mem, sc, cl, ipa, None, _mem),
        "prove: null tau": lambda: prove(f, g, None, sc, cl, ipa, None, _mem),
        "prove: null round callback": lambda: prove(f, g, _mem, None, cl, ipa, None, _mem),
        "prove: null claims callback": lambda: prove(f, g, _mem, sc, None, ipa, None, _mem),
        "prove: null ipa callback": lambda: prove(f, g, _mem, sc, cl, None, None, _mem),
        "prove: null a_hat": lambda: prove(f, g, _mem, sc, cl, ipa, None, None),
        "prove: set of the wrong curve": lambda: prove(_running(100, 90, 2, O.CURVE_VESTA)[0],
                                                       _running(1, 1, 0, O.CURVE_VESTA)[1], _mem, sc, cl, ipa, None, _mem),
        "prove: m points, not m + 1": lambda: prove(f, _running(1, 1, 0, n=128)[1], _mem, sc, cl, ipa, None, _mem),
        "prove: 1 + io > m": lambda: prove(_running(1, 1, 1)[0], g, _mem, sc, cl, ipa, None, _mem),
        "prove: 1 + io > m, m = 4": lambda: prove(_running(3, 4, 4)[0], g, _mem, sc, cl, ipa, None, _mem),
        "evaluate: null shape": lambda: _lib.load().vdfgpu_r1cs_evaluate(None, _mem, _mem, _mem),
        "evaluate: null rx": lambda: _lib.load().vdfgpu_r1cs_evaluate(s, None, _mem, _mem),
        "evaluate: null ry": lambda: _lib.load().vdfgpu_r1cs_evaluate(s, _mem, None, _mem),
        "evaluate: null output": lambda: _lib.load().vdfgpu_r1cs_evaluate(s, _mem, _mem, None),
        "evaluate: 1 + io > m": lambda: _lib.load().vdfgpu_r1cs_evaluate(_running(2, 1, 2)[2], _mem, _mem, _mem),
    }


@pytest.mark.parametrize("case", sorted(_calls()))
def test_argument_errors_launch_nothing(case):
    lib = _lib.load()
    launches = lib.vdfgpu_launch_count()
    assert _calls()[case]() == ERR_ARG, lib.vdfgpu_last_error()
    msg = lib.vdfgpu_last_error().decode()
    assert msg.startswith("running_spartan_prove" if case.startswith("prove") else "r1cs_evaluate"), msg
    assert lib.vdfgpu_launch_count() == launches
