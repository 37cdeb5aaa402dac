"""CPU: batch verification of Spartan proofs.  The device functors of the batched sparse evaluation (r1cs.cuh
EqHalfTablesBatchFn, SparseEvalBatchFn) run by a CPU loop (tests/emul/emul_spartan_verify.cpp) against
tests/spartan_ref.py; the Python batch verifier tests/spartan_verify_ref.py against the per-proof one on every
corruption; and the argument errors of vdfgpu_spartan_verify_batch and vdfgpu_r1cs_evaluate_batch, which come back
before any device work, with or without a GPU, together with the verdicts of malformed batches."""
import ctypes
import dataclasses
import random
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import pasta as O
from tests import shape_gen as S
from tests import spartan_ref as SR
from tests import spartan_verify_ref as SVR
from tests.util import aligned, ptr
from vdf_b200 import _lib
from vdf_b200 import spartan as SP

ROOT = Path(__file__).resolve().parent.parent
SZ, U32 = ctypes.c_size_t, ctypes.c_uint32
ERR_ARG = -1
FIDS = [O.FIELD_FP, O.FIELD_FQ]


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    src = ROOT / "tests" / "emul" / "emul_spartan_verify.cpp"
    lib = tmp_path_factory.mktemp("emul_spartan_verify") / "libvdf_emul_spartan_verify.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", str(lib), str(src)],
                   check=True)
    lib = ctypes.CDLL(str(lib))
    lib.emul_eq_halves.restype = ctypes.c_uint64
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


def _points(py, p, ell_x, k):
    return [[py.randrange(p) for _ in range(ell_x)] for _ in range(k)], \
           [[py.randrange(p) for _ in range(ell_x + 1)] for _ in range(k)]


# ---- the device functors on the CPU ---------------------------------------------------------------------------
@pytest.mark.parametrize("fid", FIDS)
@pytest.mark.parametrize("ell_x", [0, 1, 4, 5, 8])
def test_half_tables(emul, fid, ell_x):
    """the four half tables per proof combine into eq(r_x) and eq(r_y), whatever the parity of ell"""
    p = O.MODULUS[fid]
    py = random.Random(ell_x * 7 + fid)
    k = 3
    bits = (U32 * 4)()
    per = emul.emul_eq_halves(U32(ell_x), bits)
    assert list(bits) == [ell_x - ell_x // 2, ell_x // 2, (ell_x + 2) // 2, (ell_x + 1) // 2]
    assert per == sum(1 << b for b in bits)
    rxs, rys = _points(py, p, ell_x, k)
    out = aligned(bytes(32 * k * per))
    emul.emul_eq_half_tables(fid, SZ(k), U32(ell_x), ptr(_buf([v for r in rxs for v in r], p)),
                             ptr(_buf([v for r in rys for v in r], p)), ptr(out))
    got = _vals(out, k * per, p)
    for q in range(k):
        rec = got[q * per:(q + 1) * per]
        tabs, at = [], 0
        for b in bits:
            tabs.append(rec[at:at + (1 << b)])
            at += 1 << b
        for (hi, lo), r in (((tabs[0], tabs[1]), rxs[q]), ((tabs[2], tabs[3]), rys[q])):
            lb = len(r) // 2
            assert hi == O.eq_evals(r[:len(r) - lb], p) and lo == O.eq_evals(r[len(r) - lb:], p)
            full = O.eq_evals(r, p)
            assert [hi[i >> lb] * lo[i & ((1 << lb) - 1)] % p for i in range(1 << len(r))] == full


# (cons, vars, io): vars < m, vars = m, cons = m with io = 0, io 7 with odd ell, cons < vars with odd ell
GENERAL = [(45, 40, 7), (30, 64, 2), (64, 20, 0), (100, 90, 7), (20, 27, 7)]


def _eval_case(emul, fid, shape, k, seed):
    p = shape.m
    m = SR.padded_size(shape)
    ell_x = m.bit_length() - 1
    rxs, rys = _points(random.Random(seed), p, ell_x, k)
    row_ptr, col, val = _csr(shape)
    out = aligned(bytes(96 * k))
    emul.emul_sparse_eval_batch(fid, ptr(row_ptr), ptr(col), ptr(val), U32(shape.num_cons), U32(shape.num_vars),
                                U32(shape.num_io), SZ(k), ptr(_buf([v for r in rxs for v in r], p)),
                                ptr(_buf([v for r in rys for v in r], p)), ptr(out))
    got = _vals(out, 3 * k, p)
    want = [SR.evaluate(shape, rx, ry) for rx, ry in zip(rxs, rys)]
    assert [tuple(got[3 * q:3 * q + 3]) for q in range(k)] == want
    # one proof's values out of the batch equal that proof evaluated alone
    q = k // 2
    one = aligned(bytes(96))
    emul.emul_sparse_eval_batch(fid, ptr(row_ptr), ptr(col), ptr(val), U32(shape.num_cons), U32(shape.num_vars),
                                U32(shape.num_io), SZ(1), ptr(_buf(rxs[q], p)), ptr(_buf(rys[q], p)), ptr(one))
    assert _vals(one, 3, p) == got[3 * q:3 * q + 3]


@pytest.mark.parametrize("fid", FIDS)
@pytest.mark.parametrize("cons,vars_,io", GENERAL)
@pytest.mark.parametrize("k", [1, 3, 5])
def test_sparse_eval_batch_general_shapes(emul, fid, cons, vars_, io, k):
    """zero, +-1 and full coefficients, repeated (row, column) pairs and the heavy column of shape_gen"""
    shape = S.general_shape(fid, cons, vars_, io)
    _eval_case(emul, fid, shape, k, cons * 10 + k)


@pytest.mark.parametrize("fid", FIDS)
@pytest.mark.parametrize("t", [4, 9])
def test_sparse_eval_batch_step_shape(emul, fid, t):
    shape, _, _, _ = O.make_step_instance(fid, t, O.State(5, 6, t))
    _eval_case(emul, fid, shape, 5, t)


# ---- the Python batch verifier against the per-proof one ------------------------------------------------------
@pytest.fixture(scope="module")
def proofs():
    """three proofs of a folded step instance (u != 1, E != 0) under three transcripts, on Pallas"""
    fid, cv, p = O.FIELD_FQ, O.PALLAS, O.Q
    shape, W1, X1, _ = O.make_step_instance(fid, 4, O.State(5, 6, 4))
    _, W2, X2, _ = O.make_step_instance(fid, 4, O.State(9, 1, 4))
    r = 1 + 2 ** 100
    T = shape.cross_term(W1, 1, X1, W2, X2)
    W, E, X, u = O.fold_vec(W1, W2, r, p), [r * t % p for t in T], O.fold_vec(X1, X2, r, p), (1 + r) % p
    m = SR.padded_size(shape)
    py = random.Random(5)
    G = [cv.mul(py.randrange(1, cv.order), cv.gen) for _ in range(m + 1)]
    comm_W = cv.msm_naive(W + [0] * (m - len(W)), G[:m])
    comm_E = cv.msm_naive(E + [0] * (m - len(E)), G[:m])
    items = []
    for salt in range(3):
        tau = [py.randrange(p) for _ in range(m.bit_length() - 1)]
        pf = SR.prove(shape, W, E, u, X, tau, SR.Transcript(salt), cv, G)
        items.append((u, X, comm_W, comm_E, tau, pf))
    return shape, cv, fid, G, items


def test_reference_batch_accepts_valid_proofs(proofs):
    shape, cv, fid, G, items = proofs
    assert all(SVR.verify_one(shape, cv, fid, G, it) for it in items)
    assert SVR.verify_batch(shape, cv, fid, G, items, [3, 5, 7]) == [True] * 3


@pytest.mark.parametrize("what", SVR.CORRUPTIONS)
def test_reference_batch_rejects_exactly_the_corrupted_proof(proofs, what):
    shape, cv, fid, G, items = proofs
    bad = list(items)
    bad[1] = SVR.corrupt(items[1], what, cv, cv.order)
    one = [SVR.verify_one(shape, cv, fid, G, it) for it in bad]
    assert one == [True, False, True]
    assert SVR.verify_batch(shape, cv, fid, G, bad, [11, 13, 17]) == one


def test_reference_weights_must_be_random(proofs):
    """two openings whose errors cancel under w = (1, 1): the batch passes with those weights, not with others"""
    shape, cv, fid, G, items = proofs
    d = cv.mul(12345, cv.gen)
    a, b = list(items[0]), list(items[2])
    a[3], b[3] = cv.add(a[3], d), cv.add(b[3], cv.neg(d))   # comm_E of both: comm_a moves by +d and -d
    pair = [tuple(a), tuple(b)]
    assert not any(SVR.verify_one(shape, cv, fid, G, it) for it in pair)
    assert SVR.verify_batch(shape, cv, fid, G, pair, [1, 1]) == [True, True]
    assert SVR.verify_batch(shape, cv, fid, G, pair, [3, 5]) == [False, False]


def test_records_layout(proofs):
    """spartan_records writes the header's layout: PROOF_FES, CHAL_FES and POINTS per proof, in order"""
    shape, cv, fid, G, items = proofs
    m = SR.padded_size(shape)
    ell = m.bit_length() - 1
    from types import SimpleNamespace
    gs = SimpleNamespace(m=shape.m, num_io=shape.num_io)
    inst, pts, proof, chal = SP.spartan_records(gs, O.CURVE_PALLAS,
                                                [(u, X, O.jac_to_bytes(cv, cW), O.jac_to_bytes(cv, cE), t, pf)
                                                 for u, X, cW, cE, t, pf in items])
    k = len(items)
    assert len(inst) == 32 * k * (1 + shape.num_io)
    assert len(proof) == 32 * k * (5 * ell + 9) and len(chal) == 32 * k * (4 * ell + 6)
    assert len(pts) == 96 * k * (2 * ell + 2)
    pf = items[0][5]
    p = shape.m
    pv, cvals = O.fes_from_bytes(proof[:32 * (5 * ell + 9)], p), O.fes_from_bytes(chal[:32 * (4 * ell + 6)], p)
    assert pv[3 * ell:3 * ell + 4] == list(pf.outer_claims) and pv[-1] == pf.a_hat and pv[-3:-1] == list(pf.eval_claims)
    assert cvals[ell:2 * ell] == pf.r_x and cvals[2 * ell + 3:3 * ell + 4] == pf.r_y
    assert cvals[3 * ell + 4:3 * ell + 6] == [pf.rho, pf.u_scale] and cvals[3 * ell + 6:] == [r for _, _, r in pf.ipa]


# ---- argument errors and verdicts without a device -------------------------------------------------------------
# Without a GPU no shape or set can be built, so the handles are host structures that mirror the leading fields of
# struct vdfgpu_r1cs and vdfgpu_gens (vdf_b200/csrc/api_r1cs.cu, ctx.cuh): the checks read only those.
class _Shape(ctypes.Structure):
    _fields_ = [("field", ctypes.c_int), ("cons", ctypes.c_uint32), ("vars", ctypes.c_uint32), ("io", ctypes.c_uint32),
                ("rest", ctypes.c_uint8 * 256)]


class _Gens(ctypes.Structure):
    _fields_ = [("curve", ctypes.c_int), ("n", ctypes.c_size_t), ("rest", ctypes.c_uint8 * 256)]


_keep = []


def _handles(shape, curve=O.CURVE_PALLAS, n=None):
    m = SR.padded_size(shape)
    s = _Shape(O.FIELD_FQ, shape.num_cons, shape.num_vars, shape.num_io)
    g = _Gens(curve, m + 1 if n is None else n)
    _keep.extend((s, g))
    return ctypes.addressof(s), ctypes.addressof(g)


def _records(proofs):
    shape, cv, fid, G, items = proofs
    from types import SimpleNamespace
    gs = SimpleNamespace(m=shape.m, num_io=shape.num_io)
    return list(SP.spartan_records(gs, O.CURVE_PALLAS, [(u, X, O.jac_to_bytes(cv, cW), O.jac_to_bytes(cv, cE), t, pf)
                                                        for u, X, cW, cE, t, pf in items]))


def _call(s, g, k, rec, w, ok):
    p = _lib.as_ptr
    return _lib.load().vdfgpu_spartan_verify_batch(s, g, k, *[p(r) for r in rec], p(w), p(ok))


def _set(buf: bytes, at: int, raw32: bytes) -> bytes:
    return buf[:32 * at] + raw32 + buf[32 * (at + 1):]


def _arg_cases(proofs):
    shape, cv, fid, G, items = proofs
    k = len(items)
    m = SR.padded_size(shape)
    ell = m.bit_length() - 1
    CH = 4 * ell + 6
    s, g = _handles(shape)
    rec = _records(proofs)
    w = O.fes_to_bytes([1, 2, 3], O.Q)
    Q = O.Q.to_bytes(32, "little")
    chal = lambda at, raw: rec[:3] + [_set(rec[3], CH + at, raw)]   # noqa: E731  (proof 1's record)
    s_io = _handles(O.R1CSShape(O.Q, 3, 4, 4, [], [], []))[0]   # m = 4 < 1 + 4
    cases = {
        "null shape": (None, g, k, rec, w),
        "null set": (s, None, k, rec, w),
        "null inst": (s, g, k, [None] + rec[1:], w),
        "null points": (s, g, k, rec[:1] + [None] + rec[2:], w),
        "null proof": (s, g, k, rec[:2] + [None] + rec[3:], w),
        "null challenges": (s, g, k, rec[:3] + [None], w),
        "null weights": (s, g, k, rec, None),
        "k = 0": (s, g, 0, rec, w),
        "set of the wrong curve": (s, _handles(shape, O.CURVE_VESTA)[1], k, rec, w),
        "m points, not m + 1": (s, _handles(shape, n=m)[1], k, rec, w),
        "1 + io > m": (s_io, g, k, rec, w),
        "tau = order": (s, g, k, chal(0, Q), w),
        "r_x non-canonical": (s, g, k, chal(ell, b"\xff" * 32), w),
        "rho = order": (s, g, k, chal(3 * ell + 4, Q), w),
        "u_scale = order": (s, g, k, chal(3 * ell + 5, Q), w),
        "IPA challenge 0": (s, g, k, chal(3 * ell + 6, bytes(32)), w),
        "IPA challenge = order": (s, g, k, chal(CH - 1, Q), w),
        "weight 0": (s, g, k, rec, _set(w, 2, bytes(32))),
        "weight = order": (s, g, k, rec, _set(w, 0, Q)),
    }
    return cases


@pytest.mark.parametrize("case", ["null shape", "null set", "null inst", "null points", "null proof",
                                  "null challenges", "null weights", "k = 0", "set of the wrong curve",
                                  "m points, not m + 1", "1 + io > m", "tau = order", "r_x non-canonical",
                                  "rho = order", "u_scale = order", "IPA challenge 0", "IPA challenge = order",
                                  "weight 0", "weight = order"])
def test_argument_errors_launch_nothing(proofs, case):
    lib = _lib.load()
    s, g, k, rec, w = _arg_cases(proofs)[case]
    launches = lib.vdfgpu_launch_count()
    ok = bytearray(b"\x07" * 3)
    assert _call(s, g, k, rec, w, ok) == ERR_ARG, lib.vdfgpu_last_error()
    assert lib.vdfgpu_last_error().decode().startswith("spartan_verify_batch: ")
    assert lib.vdfgpu_launch_count() == launches
    if case not in ("null shape", "null set", "null inst", "null points", "null proof", "null challenges",
                    "null weights", "k = 0"):
        assert ok == bytes(3)   # zeroed first


def test_null_ok_is_an_argument_error(proofs):
    shape, *_ = proofs
    s, g = _handles(shape)
    rec = _records(proofs)
    assert _call(s, g, 3, rec, O.fes_to_bytes([1, 2, 3], O.Q), None) == ERR_ARG


def test_evaluate_batch_argument_errors():
    lib = _lib.load()
    mem = ctypes.create_string_buffer(1 << 12)
    s = _handles(O.R1CSShape(O.Q, 100, 90, 2, [], [], []))[0]
    s_io = _handles(O.R1CSShape(O.Q, 2, 1, 2, [], [], []))[0]
    launches = lib.vdfgpu_launch_count()
    for args in ((None, 1, mem, mem, mem), (s, 1, None, mem, mem), (s, 1, mem, None, mem), (s, 1, mem, mem, None),
                 (s, 0, mem, mem, mem), (s_io, 1, mem, mem, mem)):
        assert lib.vdfgpu_r1cs_evaluate_batch(*args) == ERR_ARG
        assert lib.vdfgpu_last_error().decode().startswith("r1cs_evaluate_batch: ")
    assert lib.vdfgpu_launch_count() == launches


def test_malformed_proofs_are_verdicts_not_errors(proofs):
    """every proof malformed in a different way: the call succeeds with verdicts 0 and no device work; a sum-check
    challenge of 0 is legal"""
    shape, cv, fid, G, items = proofs
    m = SR.padded_size(shape)
    ell = m.bit_length() - 1
    PF, CH, NP = 5 * ell + 9, 4 * ell + 6, 2 * ell + 2
    lib = _lib.load()
    s, g = _handles(shape)
    inst, pts, proof, chal = _records(proofs)
    io1 = 1 + shape.num_io
    Q, P = O.Q.to_bytes(32, "little"), O.P.to_bytes(32, "little")
    proof = _set(proof, 0 * PF + 3 * ell, Q)                 # proof 0: claim_Az = order
    inst = _set(inst, 1 * io1 + 1, Q)                        # proof 1: X[0] = order
    pt = pts[96 * 2 * NP + 96:96 * 2 * NP + 192]             # proof 2: comm_E off the curve
    y = O.fe_from_bytes(pt[32:64], O.P)
    pts = pts[:96 * 2 * NP + 96] + pt[:32] + O.fe_to_bytes(y + 1, O.P) + pt[64:] + pts[96 * 2 * NP + 192:]
    chal = _set(chal, 2 * CH + ell, bytes(32))               # a sum-check challenge of 0 (legal)
    ok = bytearray(b"\x07" * 3)
    launches = lib.vdfgpu_launch_count()
    assert _call(s, g, 3, [inst, pts, proof, chal], O.fes_to_bytes([1, 2, 3], O.Q), ok) == 0, lib.vdfgpu_last_error()
    assert ok == bytes(3)
    assert lib.vdfgpu_launch_count() == launches
    # a coordinate >= p and a non-canonical u are verdicts too
    inst2, pts2, proof2, chal2 = _records(proofs)
    pts2 = P + pts2[32:]                                     # proof 0: comm_W.X = p
    inst2 = _set(inst2, 1 * io1, b"\xff" * 32)               # proof 1: u
    proof2 = _set(proof2, 2 * PF + PF - 1, Q)                # proof 2: a_hat = order
    assert _call(s, g, 3, [inst2, pts2, proof2, chal2], O.fes_to_bytes([1, 2, 3], O.Q), ok) == 0
    assert ok == bytes(3)
    assert lib.vdfgpu_launch_count() == launches


def test_host_rejections_need_no_device(proofs):
    """proofs that fail the outer sum-check are verdicts 0 without device work, like malformed ones"""
    shape, cv, fid, G, items = proofs
    lib = _lib.load()
    s, g = _handles(shape)
    bad = [SVR.corrupt(it, what, cv, cv.order) for it, what in zip(items, ("outer round", "eval_E", "claim_Az"))]
    from types import SimpleNamespace
    gs = SimpleNamespace(m=shape.m, num_io=shape.num_io)
    rec = list(SP.spartan_records(gs, O.CURVE_PALLAS, [(u, X, O.jac_to_bytes(cv, cW), O.jac_to_bytes(cv, cE), t, pf)
                                                       for u, X, cW, cE, t, pf in bad]))
    ok = bytearray(b"\x07" * 3)
    launches = lib.vdfgpu_launch_count()
    assert _call(s, g, 3, rec, O.fes_to_bytes([1, 2, 3], O.Q), ok) == 0, lib.vdfgpu_last_error()
    assert ok == bytes(3)
    assert lib.vdfgpu_launch_count() == launches


def test_verdicts_fail_closed_when_the_call_fails(proofs):
    """three valid proofs pass the host checks, then the call fails for want of a device: no verdict may read 1.
    Runs where no CUDA device is usable; on a GPU machine the host-memory handles would reach the device work, so the
    test is skipped there."""
    lib = _lib.load()
    if lib.vdfgpu_device_count() > 0:
        pytest.skip("a CUDA device is usable: the call would not fail")
    shape, *_ = proofs
    s, g = _handles(shape)
    ok = bytearray(b"\x07" * 3)
    assert _call(s, g, 3, _records(proofs), O.fes_to_bytes([1, 2, 3], O.Q), ok) == -2, lib.vdfgpu_last_error()
    assert ok == bytes(3)
