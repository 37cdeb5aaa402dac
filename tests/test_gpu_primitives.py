"""GPU: the device primitives one operation at a time against Python integers -- the PTX carry chains of field.cuh, the
XYZZ group law of curve.cuh, the four-lane group law of quad.cuh and the batched-affine functors of msm_affine.cuh,
through the test harness tests/gpu_prims/prims.cu (never linked into libvdfgpu.so).

tests/test_emul.py runs the host branches of the same headers; the end-to-end MSM tests see a primitive only through
one final point.  Here each case is chosen for the carry, borrow or branch it reaches, and every expected value comes
from Python integers or oracle/pasta.py."""
import ctypes
import os
import random
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import pasta as O

pytestmark = pytest.mark.gpu

HERE = Path(__file__).resolve().parent
R = 1 << 256
MASK = 0xFFFFFFFF
NONE = 0xFFFFFFFF        # PAIR_NONE: the output passes its first operand through
NEG = 1 << 31            # AoS reference bit: negate the point

# field.cuh ops (FieldOp in prims.cu)
ADD, SUB, NEGF, DBL, MUL, MUL_CALL, MUL_VAL, SQR, SQR_CALL, SQR_VAL, FROM_MONT, INV, ONE, IS_CANONICAL, EQ, IS_ZERO = range(16)
# curve.cuh ops (CurveOp in prims.cu)
(C_FROM_AFFINE, C_MADD, C_MADD_CALL, C_MADD_SIGNED, C_MADD_SIGNED_CALL, C_DBL_AFFINE, C_DBL, C_ADD, C_NEG, C_FROM_JAC,
 C_TO_JAC_RAW, C_TO_JAC_NORMALISED, C_MUL_U32) = range(13)
FIELDS = [O.FIELD_FP, O.FIELD_FQ]
CURVES = [O.CURVE_PALLAS, O.CURVE_VESTA]


@pytest.fixture(scope="module")
def prims(tmp_path_factory):
    """tests/gpu_prims/libvdf_prims.so, rebuilt when prims.cu or a library header is newer (a read-only tree builds
    into a temporary directory instead)."""
    from vdf_b200 import _build
    src = HERE / "gpu_prims" / "prims.cu"
    lib = src.with_name("libvdf_prims.so")
    if not os.access(lib.parent, os.W_OK):
        lib = tmp_path_factory.mktemp("gpu_prims") / lib.name
    deps = [src] + sorted(_build.CSRC.glob("*.cuh"))
    if not lib.exists() or any(d.stat().st_mtime > lib.stat().st_mtime for d in deps):
        subprocess.run([_build._nvcc(), *_build.NVCC_FLAGS, "-shared", "-o", str(lib), str(src)], check=True)
    L = ctypes.CDLL(str(lib))
    P, SZ, I, U = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_uint32
    L.prims_field.argtypes = [I, I, P, P, P, SZ]
    L.prims_curve.argtypes = [I, I, P, P, P, P, SZ]
    L.prims_quad.argtypes = [I, I, P, P, P, SZ]
    L.prims_quad_down.argtypes = [I, P, P, SZ, I]
    L.prims_affine_batch.argtypes = [I, P, P, P, SZ, P, P, U, U, U, P, P]
    L.prims_batch_inv.argtypes = [I, P, U]
    return L


def _buf(b: bytes) -> np.ndarray:
    return np.frombuffer(bytes(b) if b else bytes(16), np.uint8).copy()


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _raw_bytes(vals) -> bytes:
    return b"".join(v.to_bytes(32, "little") for v in vals)


def _raw_list(b: bytes):
    return [int.from_bytes(b[k:k + 32], "little") for k in range(0, len(b), 32)]


# ---- field -----------------------------------------------------------------------------------------------------
def _field(prims, fid, op, A, B=None, flags=False):
    """op on raw Montgomery limb values A (and B); returns raw output values, or 0/1 flags."""
    n = len(A)
    a, b = _buf(_raw_bytes(A)), _buf(_raw_bytes(B if B is not None else A))
    out = np.zeros(n if flags else 32 * n, np.uint8)
    assert prims.prims_field(fid, op, _p(a), _p(b), _p(out), n) == 0
    return [int(x) for x in out] if flags else _raw_list(out.tobytes())


def _raw_singles(m, py):
    """Raw limb values the carry chains treat differently."""
    c = m - (1 << 254)        # the low 128 bits of m; limbs 4..6 of m are zero
    v = [0, 1, 2, m - 1, m - 2, (m - 1) // 2, (m + 1) // 2, (1 << 254) - 1, 1 << 254, R % m, MASK, 1 << 32]
    v += [(m - 1) & ~(MASK << (32 * k)) for k in range(8)]
    # limbs 4..6 zero below m's low limbs: x - m and x - y borrow out of limb 3 through the zero limbs
    v += [(1 << 254) | x for x in (0, 1, c >> 1, c - 1, (1 << 96) - 1, MASK << 64)]
    v += [1 << 127, (1 << 128) - 1, 1 << 96]
    v += [(R - 1) % m, (R - 1 - (MASK << 128)) % m]
    v += [sum((MASK if py.random() < .5 else py.randrange(1 << 32)) << (32 * k) for k in range(8)) % m
          for _ in range(200)]
    assert all(0 <= x < m for x in v)
    return v


def _raw_pairs(m, py, singles):
    """Pairs that reach each branch of add / sub, plus all pairs of the first singles and random pairs."""
    c = m - (1 << 254)
    head = singles[:40]
    A = [a for a in head for _ in head]
    B = [b for _ in head for b in head]
    for a in [1, 2, 3, m - 1, m - 2, c, 1 << 254, (m + 1) // 2] + [py.randrange(2, m - 1) for _ in range(40)]:
        for b in (m - 1 - a, m - a, m + 1 - a, a, a - 1, a + 1):           # a+b = m-1, m, m+1; a-b = 0, 1, -1
            if 0 <= b < m:
                A.append(a)
                B.append(b)
    A += [m - 1, 0, m - 1, 1]
    B += [m - 1, m - 1, 0, m - 1]                                           # a+b = 2m-2; 0 - (m-1); ...
    for x in (0, 1, c >> 1, c - 1):                                         # a+b = 2^255 + x: a+b-m borrows out of
        A.append(m - 1)                                                     # limb 3 through limbs 4..6
        B.append((1 << 255) + x - (m - 1))
    A += [py.randrange(m) for _ in range(3000)]
    B += [py.randrange(m) for _ in range(3000)]
    assert all(0 <= x < m for x in A + B)
    return A, B


@pytest.mark.parametrize("fid", FIELDS)
def test_field_binary_ops(prims, fid):
    """add, sub and the three multiplication bodies on raw values: add / sub are modular arithmetic on the limbs,
    mul is a * b * R^-1; every output is < m."""
    m = O.MODULUS[fid]
    py = random.Random(100 + fid)
    A, B = _raw_pairs(m, py, _raw_singles(m, py))
    rinv = pow(R, -1, m)
    want = {ADD: [(a + b) % m for a, b in zip(A, B)], SUB: [(a - b) % m for a, b in zip(A, B)]}
    want[MUL] = want[MUL_CALL] = want[MUL_VAL] = [a * b * rinv % m for a, b in zip(A, B)]
    for op, w in want.items():
        got = _field(prims, fid, op, A, B)
        bad = [(hex(a), hex(b)) for a, b, g, x in zip(A, B, got, w) if g != x]
        assert not bad, (op, len(bad), bad[:4])


@pytest.mark.parametrize("fid", FIELDS)
def test_field_unary_ops(prims, fid):
    """neg, dbl, the three squaring bodies, from_mont, inv (a^(m-2) in the Montgomery domain, so inv(0) = 0) and one()
    (R mod m) on raw values."""
    m = O.MODULUS[fid]
    py = random.Random(200 + fid)
    A = _raw_singles(m, py) + [py.randrange(m) for _ in range(3000)]
    rinv = pow(R, -1, m)
    want = {NEGF: [(-a) % m for a in A], DBL: [2 * a % m for a in A], FROM_MONT: [a * rinv % m for a in A],
            ONE: [R % m] * len(A)}
    want[SQR] = want[SQR_CALL] = want[SQR_VAL] = [a * a * rinv % m for a in A]
    for op, w in want.items():
        got = _field(prims, fid, op, A)
        bad = [hex(a) for a, g, x in zip(A, got, w) if g != x]
        assert not bad, (op, len(bad), bad[:4])
    inv_in = A[:300]
    assert _field(prims, fid, INV, inv_in) == [pow(a * rinv, m - 2, m) * R % m for a in inv_in]


@pytest.mark.parametrize("fid", FIELDS)
def test_field_predicates(prims, fid):
    """is_canonical on raw encodings around m (sub8_mod's borrow), eq and is_zero limb by limb."""
    m = O.MODULUS[fid]
    py = random.Random(300 + fid)
    enc = [m - 1, m, m + 1, 1 << 255, R - 1, 0, 1, (1 << 254) - 1, 1 << 254, m + (1 << 128), (1 << 254) + (1 << 128)]
    enc += [m + (1 << (32 * k)) for k in range(8)]          # m with each limb raised by one (limbs 4..6 of m are 0)
    enc += [m - (1 << (32 * k)) for k in range(8) if (m >> (32 * k)) & MASK]
    enc += [py.randrange(R) for _ in range(500)] + [py.randrange(m) for _ in range(500)]
    enc += [m + py.randrange(1 << 64) for _ in range(100)] + [m - 1 - py.randrange(1 << 64) for _ in range(100)]
    assert _field(prims, fid, IS_CANONICAL, enc, flags=True) == [int(v < m) for v in enc]
    A = [py.randrange(R) for _ in range(64)]
    A2 = list(A) + [a ^ (1 << (32 * k + py.randrange(32))) for a in A[:8] for k in range(8)]
    B2 = list(A) + [a for a in A[:8] for _ in range(8)]
    assert _field(prims, fid, EQ, A2, B2, flags=True) == [int(a == b) for a, b in zip(A2, B2)]
    Z = [0] + [1 << (32 * k + 31) for k in range(8)] + [1 << (32 * k) for k in range(8)] + A
    assert _field(prims, fid, IS_ZERO, Z, flags=True) == [int(z == 0) for z in Z]


# ---- group law ---------------------------------------------------------------------------------------------------
def _enc(vals, m) -> bytes:
    return b"".join(O.fe_to_bytes(v, m) for v in vals)


def _xyzz(cv, pt, lam=1) -> bytes:
    """XYZZ image of an affine point: X = x lam^2, Y = y lam^3, ZZ = lam^2, ZZZ = lam^3."""
    m = cv.base
    x, y = pt
    l2 = lam * lam % m
    l3 = l2 * lam % m
    return _enc([x * l2, y * l3, l2, l3], m)


def _id_zero(cv) -> bytes:
    return bytes(128)


def _id_garbage(cv, py) -> bytes:
    """The identity as ZZ = ZZZ = 0 with arbitrary X and Y: the contract is identity <=> ZZ == 0."""
    return _enc([py.randrange(1, cv.base), py.randrange(1, cv.base), 0, 0], cv.base)


def _aff(cv, pt) -> bytes:
    return bytes(64) if pt is None else _enc(pt, cv.base)


def _dec_xyzz(cv, b: bytes):
    """XYZZ bytes -> affine point or None; checks canonical limbs, ZZ^3 = ZZZ^2 and that the point is on the curve."""
    m = cv.base
    X, Y, ZZ, ZZZ = (O.fe_from_bytes(b[k:k + 32], m) for k in range(0, 128, 32))
    if ZZ == 0:
        return None
    assert pow(ZZ, 3, m) == pow(ZZZ, 2, m), "ZZ^3 != ZZZ^2"
    pt = (X * pow(ZZ, -1, m) % m, Y * pow(ZZZ, -1, m) % m)
    assert cv.on_curve(pt)
    return pt


def _dec_jac(cv, b: bytes):
    m = cv.base
    X, Y, Z = (O.fe_from_bytes(b[k:k + 32], m) for k in range(0, 96, 32))
    if Z == 0:
        assert b == bytes(96), "identity must be (0, 0, 0)"
        return None
    pt = cv.jac_to_affine((X, Y, Z))
    assert cv.on_curve(pt)
    return pt


def _curve(prims, cid, op, a, b=None, aux=None, n=None):
    """op over n elementwise inputs: a, b concatenated encodings, aux a list of u32."""
    size_out = 96 if op in (C_TO_JAC_RAW, C_TO_JAC_NORMALISED) else 128
    ba = _buf(a)
    bb = _buf(b) if b is not None else None
    bx = np.array(aux, np.uint32) if aux is not None else None
    out = np.zeros(size_out * n, np.uint8)
    assert prims.prims_curve(cid, op, _p(ba), _p(bb), _p(bx), _p(out), n) == 0
    return [out.tobytes()[size_out * k:size_out * (k + 1)] for k in range(n)]


def _rand_pt(cv, py):
    return cv.mul(py.randrange(1, cv.order), cv.gen)


def _lam(cv, py):
    return py.randrange(2, cv.base)


def _add_cases(cv, py, npts=3):
    """(acc, q) as XYZZ bytes and the oracle's acc + q: acc in {identity (both forms), P, P with another ZZ, -P,
    unrelated Q} against q = P, plus q = identity (both forms).  lambda = 1 and random lambdas."""
    accs, qs, want = [], [], []
    for k in range(npts):
        P, Q = _rand_pt(cv, py), _rand_pt(cv, py)
        lq = 1 if k == 0 else _lam(cv, py)
        q = _xyzz(cv, P, lq)
        for acc, pt in ((_id_zero(cv), None), (_id_garbage(cv, py), None), (_xyzz(cv, P, 1), P),
                        (_xyzz(cv, P, _lam(cv, py)), P), (_xyzz(cv, cv.neg(P), _lam(cv, py)), cv.neg(P)),
                        (_xyzz(cv, cv.neg(P), 1), cv.neg(P)), (_xyzz(cv, Q, _lam(cv, py)), Q), (_xyzz(cv, Q, 1), Q)):
            accs.append(acc)
            qs.append(q)
            want.append(cv.add(pt, P))
        for qi in (_id_zero(cv), _id_garbage(cv, py)):
            accs.append(_xyzz(cv, P, _lam(cv, py)))
            qs.append(qi)
            want.append(P)
    return accs, qs, want


@pytest.mark.parametrize("cid", CURVES)
def test_curve_add_and_madd(prims, cid):
    """Curve::add and the four mixed additions against the oracle, every special case: identity accumulators with
    ZZ = 0 and non-zero X / Y, the same point with a different ZZ (doubling), -P (cancellation), identity operands."""
    cv = O.CURVES[cid]
    py = random.Random(400 + cid)
    accs, qs, want = _add_cases(cv, py)
    n = len(accs)
    got = _curve(prims, cid, C_ADD, b"".join(accs), b"".join(qs), n=n)
    assert [_dec_xyzz(cv, g) for g in got] == want
    # mixed: the affine operand of every case whose q is not the identity
    keep = [k for k, q in enumerate(qs) if _dec_xyzz(cv, q) is not None]
    acc = b"".join(accs[k] for k in keep)
    P = [_dec_xyzz(cv, qs[k]) for k in keep]
    aff = b"".join(_aff(cv, p) for p in P)
    for op in (C_MADD, C_MADD_CALL):
        got = _curve(prims, cid, op, acc, aff, n=len(keep))
        assert [_dec_xyzz(cv, g) for g in got] == [want[k] for k in keep], op
    # signed: negate on and off, and the affine identity (0, 0) (a no-op either way)
    accs2 = [accs[k] for k in keep] * 4
    ops2 = [p for p in P] * 2 + [None] * (2 * len(keep))
    neg2 = [0] * len(keep) + [1] * len(keep) + [0] * len(keep) + [1] * len(keep)
    want2 = []
    for a, p, ng in zip(accs2, ops2, neg2):
        want2.append(cv.add(_dec_xyzz(cv, a), cv.neg(p) if ng else p))
    for op in (C_MADD_SIGNED, C_MADD_SIGNED_CALL):
        got = _curve(prims, cid, op, b"".join(accs2), b"".join(_aff(cv, p) for p in ops2), neg2, n=len(accs2))
        assert [_dec_xyzz(cv, g) for g in got] == want2, op


@pytest.mark.parametrize("cid", CURVES)
def test_curve_dbl_neg_and_conversions(prims, cid):
    """dbl, dbl_affine, neg, from_affine, the Jacobian conversions and mul_u32 against the oracle."""
    cv = O.CURVES[cid]
    m = cv.base
    py = random.Random(500 + cid)
    pts = [_rand_pt(cv, py) for _ in range(6)]
    xs = [_xyzz(cv, p, 1 if k == 0 else _lam(cv, py)) for k, p in enumerate(pts)] + [_id_zero(cv), _id_garbage(cv, py)]
    ref = pts + [None, None]
    n = len(xs)
    assert [_dec_xyzz(cv, g) for g in _curve(prims, cid, C_DBL, b"".join(xs), n=n)] == [cv.add(p, p) for p in ref]
    assert [_dec_xyzz(cv, g) for g in _curve(prims, cid, C_NEG, b"".join(xs), n=n)] == [cv.neg(p) for p in ref]
    aff = b"".join(_aff(cv, p) for p in pts)
    assert [_dec_xyzz(cv, g) for g in _curve(prims, cid, C_DBL_AFFINE, aff, n=len(pts))] == [cv.add(p, p) for p in pts]
    got = _curve(prims, cid, C_FROM_AFFINE, aff + bytes(64), n=len(pts) + 1)
    assert [_dec_xyzz(cv, g) for g in got] == pts + [None]
    assert got[-1] == bytes(128)
    # Jacobian in: Z = 0 with garbage X / Y, Z = 1, random Z
    jac, jref = [], []
    for k, p in enumerate(pts):
        Z = [0, 1, py.randrange(2, m)][k % 3]
        if Z == 0:
            jac.append(_enc([py.randrange(1, m), py.randrange(1, m), 0], m))
            jref.append(None)
        else:
            jac.append(_enc([p[0] * Z * Z, p[1] * Z * Z * Z, Z], m))
            jref.append(p)
    assert [_dec_xyzz(cv, g) for g in _curve(prims, cid, C_FROM_JAC, b"".join(jac), n=len(jac))] == jref
    # Jacobian out: raw (as group elements, the identity as (0, 0, 0)) and normalised (byte for byte)
    assert [_dec_jac(cv, g) for g in _curve(prims, cid, C_TO_JAC_RAW, b"".join(xs), n=n)] == ref
    assert _curve(prims, cid, C_TO_JAC_NORMALISED, b"".join(xs), n=n) == [O.jac_to_bytes(cv, p) for p in ref]
    # mul_u32
    ks = [0, 1, 2, 3, 1 << 31, MASK, py.randrange(1 << 32), py.randrange(1 << 16)]
    mx = [x for x in xs for _ in ks]
    mk = [k for _ in xs for k in ks]
    got = _curve(prims, cid, C_MUL_U32, b"".join(mx), aux=mk, n=len(mx))
    assert [_dec_xyzz(cv, g) for g in got] == [cv.mul(k, p) for p in ref for k in mk[:len(ks)]]


# ---- quad --------------------------------------------------------------------------------------------------------
def _quad(prims, cid, op, accs, qs):
    n = len(accs)
    out = np.zeros(128 * n, np.uint8)
    assert prims.prims_quad(cid, op, _p(_buf(b"".join(accs))), _p(_buf(b"".join(qs))), _p(out), n) == 0
    return [out.tobytes()[128 * k:128 * (k + 1)] for k in range(n)]


@pytest.mark.parametrize("cid", CURVES)
def test_quad_add_and_dbl(prims, cid):
    """Quad<F>::add / dbl on five warps (eight quads each, in blocks of two warps), every warp mixing all branches in
    one call: early return on an identity q, identity acc (both forms), doubling, cancellation, generic additions.
    Same group elements as Curve<F>::add / dbl and the oracle, ZZ^3 = ZZZ^2."""
    cv = O.CURVES[cid]
    py = random.Random(600 + cid)
    accs, qs, want = [], [], []
    for w in range(5):
        P, Q = _rand_pt(cv, py), _rand_pt(cv, py)
        lp = 1 if w == 0 else _lam(cv, py)
        case = [
            (_xyzz(cv, P, _lam(cv, py)), _id_zero(cv), P),                                      # q identity
            (_xyzz(cv, P, lp), _id_garbage(cv, py), P),
            (_id_zero(cv), _xyzz(cv, P, lp), P),                                                # acc identity
            (_id_garbage(cv, py), _xyzz(cv, P, _lam(cv, py)), P),
            (_xyzz(cv, P, _lam(cv, py)), _xyzz(cv, P, lp), cv.add(P, P)),                       # doubling
            (_xyzz(cv, cv.neg(P), _lam(cv, py)), _xyzz(cv, P, lp), None),                       # cancellation
            (_xyzz(cv, Q, _lam(cv, py)), _xyzz(cv, P, lp), cv.add(Q, P)),                       # generic
            (_xyzz(cv, Q, 1), _xyzz(cv, P, _lam(cv, py)), cv.add(Q, P)),
        ]
        case = case[w:] + case[:w]          # each branch at a different quad of its warp from warp to warp
        for a, q, r in case:
            accs.append(a)
            qs.append(q)
            want.append(r)
    got = _quad(prims, cid, 0, accs, qs)
    assert [_dec_xyzz(cv, g) for g in got] == want
    flat = _curve(prims, cid, C_ADD, b"".join(accs), b"".join(qs), n=len(accs))
    assert [_dec_xyzz(cv, g) for g in flat] == want
    # doubling: a point, its negation, the identity in both forms, in every warp
    dacc, dwant = [], []
    for w in range(3):
        P, Q = _rand_pt(cv, py), _rand_pt(cv, py)
        row = [(_xyzz(cv, P, _lam(cv, py)), P), (_xyzz(cv, cv.neg(P), _lam(cv, py)), cv.neg(P)),
               (_id_zero(cv), None), (_id_garbage(cv, py), None), (_xyzz(cv, P, 1), P), (_xyzz(cv, Q, 1), Q),
               (_id_garbage(cv, py), None), (_xyzz(cv, Q, _lam(cv, py)), Q)]
        for a, p in row[w:] + row[:w]:
            dacc.append(a)
            dwant.append(cv.add(p, p))
    got = _quad(prims, cid, 1, dacc, dacc)
    assert [_dec_xyzz(cv, g) for g in got] == dwant
    flat = _curve(prims, cid, C_DBL, b"".join(dacc), n=len(dacc))
    assert [_dec_xyzz(cv, g) for g in flat] == dwant


@pytest.mark.parametrize("cid", CURVES)
def test_quad_down(prims, cid):
    """Quad<F>::down(v, delta) returns the point held `delta` lanes up, byte for byte, for every lane whose source lane
    is inside its warp (two warps)."""
    py = random.Random(700 + cid)
    lanes = [bytes(py.randrange(256) for _ in range(128)) for _ in range(64)]
    for delta in (4, 8, 16):
        out = np.zeros(128 * 64, np.uint8)
        assert prims.prims_quad_down(cid, _p(_buf(b"".join(lanes))), _p(out), 64, delta) == 0
        got = [out.tobytes()[128 * k:128 * (k + 1)] for k in range(64)]
        for i in range(64):
            if i % 32 + delta < 32:
                assert got[i] == lanes[i + delta], (delta, i)


# ---- batched affine ----------------------------------------------------------------------------------------------
KINDS = ("ADD", "DBL", "TAKE1", "TAKE2", "ZERO", "NONE")


def _affine_table(cv, py):
    """Points of the AoS table: six distinct points, the identity (0, 0) at 6, a copy of point 0 at 7, -point 1 at 8;
    and reference pairs of each kind (bit 31 = negate)."""
    pts = [_rand_pt(cv, py) for _ in range(6)] + [None]
    pts += [pts[0], cv.neg(pts[1])]
    I = 6
    pairs = {
        "ADD": [(0, 2), (3, 4 | NEG), (5 | NEG, 1), (2 | NEG, 3 | NEG), (7, 1)],
        "DBL": [(0, 0), (0, 7), (1 | NEG, 1 | NEG), (1, 8 | NEG), (8, 8)],
        "TAKE1": [(2, I), (3 | NEG, I | NEG), (8, I)],
        "TAKE2": [(I, 4), (I | NEG, 5 | NEG), (I, I), (I | NEG, I)],
        "ZERO": [(0, 0 | NEG), (1, 8), (7 | NEG, 0), (4 | NEG, 4)],
        "NONE": [(3, NONE), (I | NEG, NONE), (2 | NEG, NONE), (I, NONE)],
    }
    return pts, pairs


def _affine_layout(T, K, M, rot):
    """Kind of every output: thread t owns outputs t, t + T, ... (at most K).  Position j of a chain of length cnt
    gets kind (t + rot + j) mod 6, its last position (t + rot + 3) mod 6, so over six threads (or six rotations)
    every kind is first, in the middle and last of some chain."""
    kinds = [None] * M
    for t in range(min(T, M)):
        chain = list(range(t, M, T))[:K]
        for j, o in enumerate(chain):
            kinds[o] = (t + rot + (3 if j == len(chain) - 1 and j > 0 else j)) % 6
    assert None not in kinds
    return kinds


def _affine_run(prims, cid, pts, ra, rb, T, K, aos):
    cv = O.CURVES[cid]
    m = cv.base
    M = len(ra)
    if aos:
        src = _buf(b"".join(_aff(cv, p) for p in pts))
        xs = ys = None
        refs_a, refs_b = ra, rb
    else:   # SoA has no negation bit: negated points are stored after the table
        table = pts + [cv.neg(p) for p in pts]
        src = None
        xs = _buf(_enc([0 if p is None else p[0] for p in table], m))
        ys = _buf(_enc([0 if p is None else p[1] for p in table], m))
        soa = lambda r: r if r == NONE else (r & ~NEG) + (len(pts) if r & NEG else 0)   # noqa: E731
        refs_a, refs_b = [soa(r) for r in ra], [soa(r) for r in rb]
    ox, oy = np.zeros(32 * M, np.uint8), np.zeros(32 * M, np.uint8)
    npts = 2 * len(pts)
    assert prims.prims_affine_batch(cid, _p(src), _p(xs), _p(ys), npts if not aos else len(pts),
                                    _p(np.array(refs_a, np.uint32)), _p(np.array(refs_b, np.uint32)), M, T, K,
                                    _p(ox), _p(oy)) == 0
    X, Y = O.fes_from_bytes(ox.tobytes(), m), O.fes_from_bytes(oy.tobytes(), m)
    assert all(v < m for v in _raw_list(ox.tobytes()) + _raw_list(oy.tobytes()))
    return [None if x == 0 and y == 0 else (x, y) for x, y in zip(X, Y)]


@pytest.mark.parametrize("cid", CURVES)
def test_affine_batch_mixed_pair_kinds(prims, cid):
    """AffineFwdFn -> BatchInvFn -> AffineBwdFn on caller-built pair lists with every PairKind (ADD, DBL, TAKE1,
    TAKE2, ZERO and pass-through) at the first, a middle and the last position of one thread's chain, T = 1 and
    T > 1 (more than one block), K not dividing the output count; AoS (gather path, bit-31 negation, -(0, 0) stays
    the identity) and SoA reads.  Every output is the oracle's sum: exceptional pairs never poison a batch."""
    cv = O.CURVES[cid]
    py = random.Random(800 + cid)
    pts, pairs = _affine_table(cv, py)
    pt = lambda r: None if r == NONE else (cv.neg(pts[r & ~NEG]) if r & NEG else pts[r])   # noqa: E731
    for name, lst in pairs.items():   # the table says what it means
        for a, b in lst:
            A, B = pt(a), pt(b)
            kind = ("NONE" if b == NONE else "TAKE2" if A is None else "TAKE1" if B is None else
                    "ADD" if A[0] != B[0] else "DBL" if A[1] == B[1] else "ZERO")
            assert kind == name, (name, a, b)
    seen = set()
    configs = [(1, 16, 13, rot) for rot in range(6)] + [(6, 5, 28, 0), (13, 4, 50, 0), (40, 7, 270, 0), (150, 3, 449, 0)]
    for T, K, M, rot in configs:
        assert M <= T * K
        kinds = _affine_layout(T, K, M, rot)
        use = {k: 0 for k in range(6)}
        ra, rb = [], []
        for o, kd in enumerate(kinds):
            lst = pairs[KINDS[kd]]
            a, b = lst[(use[kd] + o) % len(lst)]
            use[kd] += 1
            ra.append(a)
            rb.append(b)
            cnt = len(range(o % T, M, T)[:K])
            j = o // T
            seen.add((kd, "first" if j == 0 else "last" if j == cnt - 1 else "middle"))
        want = [pt(a) if b == NONE else cv.add(pt(a), pt(b)) for a, b in zip(ra, rb)]
        for aos in (True, False):
            got = _affine_run(prims, cid, pts, ra, rb, T, K, aos)
            bad = [(o, KINDS[kinds[o]]) for o in range(M) if got[o] != want[o]]
            assert not bad, (T, K, M, rot, aos, bad[:6])
    assert seen == {(k, p) for k in range(6) for p in ("first", "middle", "last")}


@pytest.mark.parametrize("fid", FIELDS)
def test_batch_inv(prims, fid):
    """BatchInvFn on its own around J = 32 elements per thread: n = 1, 31, 32, 33, 64, 65, 1000."""
    m = O.MODULUS[fid]
    py = random.Random(900 + fid)
    for n in (1, 31, 32, 33, 64, 65, 1000):
        vals = [1, m - 1, 2, (m + 1) // 2] + [py.randrange(1, m) for _ in range(n)]
        vals = vals[:n]
        v = _buf(_enc(vals, m))
        assert prims.prims_batch_inv(fid, _p(v), n) == 0
        assert _raw_list(v.tobytes()) == [O.to_mont(pow(x, -1, m), m) for x in vals], n
