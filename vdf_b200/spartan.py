"""Host-side mirror of the sum-check building blocks of CompressedSNARK::prove (src/nova/proof.rs:360-368 -> nova-snark
0.8 spartan_with_ipa_pc: EqPolynomial::evals, SumcheckProof::{prove_cubic_with_additive_term, prove_quad},
MultilinearPolynomial::{bound_poly_var_top, evaluate}).  The arithmetic runs on the GPU through the C ABI; the
transcript (round polynomial in, challenge out) is the caller's, passed as a Python callable."""
from __future__ import annotations

import ctypes
from typing import Callable, List, Sequence, Tuple

from . import _lib
from .encoding import MODULUS, fe_from_bytes, fe_to_bytes, fes_from_bytes, fes_to_bytes

Challenge = Callable[[int, Tuple[int, ...]], int]


def eq_evals(field_id: int, r: Sequence[int]) -> List[int]:
    m = MODULUS[field_id]
    out = bytearray(32 << len(r))
    _lib.check(_lib.load().vdfgpu_eq_evals(field_id, _lib.as_ptr(fes_to_bytes(r, m) or bytes(32)), len(r), _lib.as_ptr(out)))
    return fes_from_bytes(bytes(out), m)


def poly_evaluate(field_id: int, poly: Sequence[int], r: Sequence[int]) -> int:
    m = MODULUS[field_id]
    if len(poly) != 1 << len(r):
        raise ValueError("poly_evaluate: the table must have 2^len(r) entries")
    out = bytearray(32)
    _lib.check(_lib.load().vdfgpu_poly_evaluate(field_id, _lib.as_ptr(fes_to_bytes(poly, m)), _lib.as_ptr(fes_to_bytes(r, m) or bytes(32)),
                                                len(r), _lib.as_ptr(out)))
    return fe_from_bytes(bytes(out), m)


def _round_trampoline(m: int, challenge: Challenge, log: list):
    def fn(_user, rnd, evals_ptr, n_evals, r_out):
        try:
            raw = ctypes.string_at(evals_ptr, 32 * n_evals)
            evals = tuple(fes_from_bytes(raw, m))
            r = challenge(int(rnd), evals) % m
            log.append((evals, r))
            ctypes.memmove(r_out, fe_to_bytes(r, m), 32)
            return 0
        except Exception:   # surfaces as VDFGPU_ERR_STATE
            return 1
    return _lib.ROUND_FN(fn)


def sumcheck(field_id: int, tables: Sequence[Sequence[int]], challenge: Challenge):
    """Cubic-with-additive-term sum-check over 4 tables (comb = A (B C - D)) or quadratic over 2 (comb = A B).
    Returns (per-round evaluations, challenges, final evaluations)."""
    m = MODULUS[field_id]
    n = len(tables[0])
    ell = n.bit_length() - 1
    if n != 1 << ell or any(len(t) != n for t in tables) or len(tables) not in (2, 4):
        raise ValueError("sumcheck: 2 or 4 tables of the same power-of-two length")
    lib = _lib.load()
    bufs = [fes_to_bytes(t, m) for t in tables]
    log: list = []
    cb = _round_trampoline(m, challenge, log)
    final = bytearray(32 * len(tables))
    cbp = ctypes.cast(cb, ctypes.c_void_p)
    if len(tables) == 4:
        rc = lib.vdfgpu_sumcheck_cubic(field_id, *[_lib.as_ptr(b) for b in bufs], ell, cbp, None, _lib.as_ptr(final))
    else:
        rc = lib.vdfgpu_sumcheck_quad(field_id, *[_lib.as_ptr(b) for b in bufs], ell, cbp, None, _lib.as_ptr(final))
    _lib.check(rc)
    return [e for e, _ in log], [r for _, r in log], fes_from_bytes(bytes(final), m)


# ---- inner-product-argument building blocks -----------------------------------------------------------------
def vec_lincomb(field_id: int, a: Sequence[int], b: Sequence[int], x: int, y: int) -> List[int]:
    """out[i] = x a[i] + y b[i] (the vector folds of one IPA round)."""
    m = MODULUS[field_id]
    if len(a) != len(b):
        raise ValueError("vec_lincomb: length mismatch")
    out = bytearray(32 * len(a))
    _lib.check(_lib.load().vdfgpu_vec_lincomb(field_id, _lib.as_ptr(fes_to_bytes(a, m)), _lib.as_ptr(fes_to_bytes(b, m)), len(a),
                                              _lib.as_ptr(fe_to_bytes(x, m)), _lib.as_ptr(fe_to_bytes(y, m)), _lib.as_ptr(out)))
    return fes_from_bytes(bytes(out), m)


def inner_product(field_id: int, a: Sequence[int], b: Sequence[int]) -> int:
    m = MODULUS[field_id]
    if len(a) != len(b):
        raise ValueError("inner_product: length mismatch")
    out = bytearray(32)
    _lib.check(_lib.load().vdfgpu_inner_product(field_id, _lib.as_ptr(fes_to_bytes(a, m) or bytes(32)),
                                                _lib.as_ptr(fes_to_bytes(b, m) or bytes(32)), len(a), _lib.as_ptr(out)))
    return fe_from_bytes(bytes(out), m)


def points_lincomb(curve: int, P: bytes, Q: bytes, w1: int, w2: int) -> bytes:
    """out[i] = w1 P[i] + w2 Q[i] on 72-byte affine points (CommitGens::fold of one IPA round)."""
    from .encoding import CURVE_ORDER
    if len(P) != len(Q) or len(P) % 72:
        raise ValueError("points_lincomb: two affine arrays of the same length")
    order = CURVE_ORDER[curve]
    out = bytearray(len(P))
    _lib.check(_lib.load().vdfgpu_points_lincomb(curve, _lib.as_ptr(P), _lib.as_ptr(Q), len(P) // 72,
                                                 _lib.as_ptr(fe_to_bytes(w1, order)), _lib.as_ptr(fe_to_bytes(w2, order)), _lib.as_ptr(out)))
    return bytes(out)



# ---- the whole inner-product argument on a resident generator set -----------------------------------------------
IpaChallenge = Callable[[int, bytes, bytes], int]


def _ipa_trampoline(order: int, challenge: IpaChallenge, log: list):
    def fn(_user, rnd, L_ptr, R_ptr, r_out):
        try:
            L, R = ctypes.string_at(L_ptr, 96), ctypes.string_at(R_ptr, 96)
            r = challenge(int(rnd), L, R) % order
            log.append((L, R, r))
            ctypes.memmove(r_out, fe_to_bytes(r, order), 32)
            return 0
        except Exception:   # surfaces as VDFGPU_ERR_STATE
            return 1
    return _lib.IPA_ROUND_FN(fn)


def _ipa_call(gens, fn_name: str, a_arg, b_arg, ell: int, u_scale: int, challenge: IpaChallenge):
    from .encoding import CURVE_ORDER
    order = CURVE_ORDER[gens.curve]
    log: list = []
    cb = _ipa_trampoline(order, challenge, log)
    a_hat = bytearray(32)
    _lib.check(getattr(_lib.load(), fn_name)(gens._h, a_arg, b_arg, ell, _lib.as_ptr(fe_to_bytes(u_scale, order)),
                                             ctypes.cast(cb, ctypes.c_void_p), None, _lib.as_ptr(a_hat)))
    return [L for L, _, _ in log], [R for _, R, _ in log], [r for _, _, r in log], fe_from_bytes(bytes(a_hat), order)


def ipa_prove(gens, a: Sequence[int], b: Sequence[int], u_scale: int, challenge: IpaChallenge):
    """The inner-product argument over 2^ell-entry vectors a, b on the resident set `gens` (at least 2^ell + 1 points;
    U = u_scale * gens[2^ell]).  challenge(round, L, R) is the caller's transcript: it receives the round's commitments
    as 96-byte normalised points and returns r != 0.  Returns (L list, R list, challenges, a_hat)."""
    from .encoding import CURVE_ORDER
    order = CURVE_ORDER[gens.curve]
    n = len(a)
    ell = n.bit_length() - 1
    if n != 1 << ell or len(b) != n:
        raise ValueError("ipa_prove: a and b need the same power-of-two length")
    return _ipa_call(gens, "vdfgpu_ipa_prove", _lib.as_ptr(fes_to_bytes(a, order)), _lib.as_ptr(fes_to_bytes(b, order)),
                     ell, u_scale, challenge)


def ipa_prove_dev(gens, a_dev, b_dev, u_scale: int, challenge: IpaChallenge):
    """ipa_prove on device vectors (CUDA tensors of 32-byte Montgomery elements, consumed) on the calling thread's
    stream."""
    nbytes = a_dev.numel() * a_dev.element_size()
    n = nbytes // 32
    ell = n.bit_length() - 1
    if nbytes % 32 or n != 1 << ell or b_dev.numel() * b_dev.element_size() != nbytes:
        raise ValueError("ipa_prove_dev: a and b need the same power-of-two number of elements")
    return _ipa_call(gens, "vdfgpu_ipa_prove_dev", a_dev.data_ptr(), b_dev.data_ptr(), ell, u_scale, challenge)


def ipa_gens_hat(gens, r: Sequence[int]) -> bytes:
    """The verifier's folded generator G_hat = <s, gens[0, 2^len(r))> as a 96-byte normalised point."""
    from .encoding import CURVE_ORDER
    order = CURVE_ORDER[gens.curve]
    out = bytearray(96)
    _lib.check(_lib.load().vdfgpu_ipa_gens_hat(gens._h, _lib.as_ptr(fes_to_bytes(r, order) or bytes(32)), len(r),
                                               _lib.as_ptr(out)))
    return bytes(out)


# ---- verification of inner-product arguments ---------------------------------------------------------------------
# A proof as the verifier receives it: what ipa_prove returns (L list, R list, challenges, a_hat) and the instance
# (comm_a as a 96-byte point, c = <a, b>, b_hat = <b, s>, u_scale).
IpaProof = Tuple[Sequence[bytes], Sequence[bytes], Sequence[int], int, bytes, int, int, int]


def ipa_b_hat(field_id: int, rs: Sequence[int], terms: Sequence[Tuple[int, Sequence[int]]]) -> int:
    """b_hat = <b, s> for b = sum_i rho_i eq(x_i), terms = [(rho_i, x_i)], in closed form: <eq(x), s> =
    prod_j ((1 - x_j) r_j^-1 + x_j r_j).  An x shorter than rs stands for an eq table zero-padded at the top (eq over
    x with leading zero coordinates)."""
    m = MODULUS[field_id]
    inv = [pow(r, -1, m) for r in rs]
    out = 0
    for rho, x in terms:
        if len(x) > len(rs):
            raise ValueError("ipa_b_hat: a point has more coordinates than there are challenges")
        x = [0] * (len(rs) - len(x)) + list(x)
        v = rho % m
        for xj, r, ri in zip(x, rs, inv):
            v = v * ((1 - xj) * ri + xj * r) % m
        out = (out + v) % m
    return out


def ipa_verify_batch(gens, proofs: Sequence[IpaProof], weights: Sequence[int] | None = None) -> List[bool]:
    """Verifies inner-product arguments over the resident set `gens` (at least 2^ell + 1 points) in one call, one
    verdict per proof.  All proofs need the same ell.  weights: one non-zero weight per proof for the random linear
    combination; None draws them with `secrets`.  A caller that passes its own must draw them uniformly and out of
    the provers' sight: predictable weights let two invalid proofs cancel."""
    import secrets

    from .encoding import CURVE_ORDER
    order = CURVE_ORDER[gens.curve]
    k = len(proofs)
    if k == 0:
        return []
    ell = len(proofs[0][2])
    if any(len(p[0]) != ell or len(p[1]) != ell or len(p[2]) != ell for p in proofs):
        raise ValueError("ipa_verify_batch: every proof needs ell L, R and challenges, the same ell for all")
    if any(len(x) != 96 for p in proofs for x in (p[4], *p[0], *p[1])):
        raise ValueError("ipa_verify_batch: comm_a, L and R must be 96-byte Jacobian points")
    if weights is None:
        weights = [1 + secrets.randbelow(order - 1) for _ in range(k)]
    if len(weights) != k:
        raise ValueError("ipa_verify_batch: one weight per proof")
    comm = b"".join(p[4] for p in proofs)
    Ls = b"".join(x for p in proofs for x in p[0]) or bytes(96)
    Rs = b"".join(x for p in proofs for x in p[1]) or bytes(96)
    rs = fes_to_bytes([r for p in proofs for r in p[2]], order) or bytes(32)
    col = lambda i: _lib.as_ptr(fes_to_bytes([p[i] for p in proofs], order))  # noqa: E731
    ok = bytearray(k)
    _lib.check(_lib.load().vdfgpu_ipa_verify_batch(gens._h, ell, k, _lib.as_ptr(comm), _lib.as_ptr(Ls), _lib.as_ptr(Rs),
                                                   _lib.as_ptr(rs), col(3), col(5), col(6), col(7),
                                                   _lib.as_ptr(fes_to_bytes(weights, order)), _lib.as_ptr(ok)))
    return [bool(v) for v in ok]


# ---- Spartan of a resident running instance (RelaxedR1CSSNARK::prove [R], nova.RunningProver.spartan_prove) ----------
SPARTAN_OUTER, SPARTAN_EVAL, SPARTAN_IPA = 0, 1, 2


def padded_layout(num_cons: int, num_vars: int, num_io: int) -> Tuple[int, Callable[[int], int]]:
    """nova's R1CSShape::pad [R]: m = the next power of two >= max(num_vars, num_cons), and the padded column of the
    shape's column c (c if c < num_vars, else c + m - num_vars): W occupies [0, m), u is column m, X starts at m + 1, and
    z has 2m entries.  The library requires 1 + num_io <= m."""
    need = max(num_cons, num_vars, 1)
    m = 1 << (need - 1).bit_length()
    return m, lambda c: c if c < num_vars else c + m - num_vars


def _value_bytes(v, m: int) -> bytes:
    """a callback's answer as the library reads it: an integer (reduced, canonical), or 32 raw bytes passed as they are"""
    if isinstance(v, (bytes, bytearray)):
        if len(v) != 32:
            raise ValueError("a raw value is 32 bytes")
        return bytes(v)
    return fe_to_bytes(v, m)


def spartan_trampolines(m: int, transcript, log: list):
    """The three C callbacks of vdfgpu_running_spartan_prove around a Python transcript object with sumcheck_round(rnd,
    evals), claims(stage, values) and ipa_round(rnd, L, R); each answer is an integer or 32 raw bytes.  Every call is
    appended to log as ("round", evals, r), ("claims", stage, values, answers) or ("ipa", L, R, r), answers as the
    library decodes them.  m: the shape's field, which is the IPA set's scalar field.  An exception in the transcript
    surfaces as VDFGPU_ERR_STATE."""
    def sc(_user, rnd, evals_ptr, n_evals, r_out):
        try:
            evals = tuple(fes_from_bytes(ctypes.string_at(evals_ptr, 32 * n_evals), m))
            raw = _value_bytes(transcript.sumcheck_round(int(rnd), evals), m)
            log.append(("round", evals, fe_from_bytes(raw, m)))
            ctypes.memmove(r_out, raw, 32)
            return 0
        except Exception:
            return 1

    def claims(_user, stage, in_ptr, n_in, out_ptr, n_out):
        try:
            vals = tuple(fes_from_bytes(ctypes.string_at(in_ptr, 32 * n_in), m))
            ans = list(transcript.claims(int(stage), vals))
            if len(ans) != n_out:
                raise ValueError("claims: wrong number of answers")
            raw = b"".join(_value_bytes(v, m) for v in ans)
            log.append(("claims", int(stage), vals, tuple(fes_from_bytes(raw, m))))
            ctypes.memmove(out_ptr, raw, 32 * n_out)
            return 0
        except Exception:
            return 1

    def ipa(_user, rnd, L_ptr, R_ptr, r_out):
        try:
            L, R = ctypes.string_at(L_ptr, 96), ctypes.string_at(R_ptr, 96)
            raw = _value_bytes(transcript.ipa_round(int(rnd), L, R), m)
            log.append(("ipa", L, R, fe_from_bytes(raw, m)))
            ctypes.memmove(r_out, raw, 32)
            return 0
        except Exception:
            return 1
    return _lib.ROUND_FN(sc), _lib.CLAIMS_FN(claims), _lib.IPA_ROUND_FN(ipa)


# ---- verification of Spartan proofs in batches (RelaxedR1CSSNARK::verify [R], vdfgpu_spartan_verify_batch) -----------
# An item as the verifier holds it: the instance (u, X, comm_W, comm_E; commitments as affine tuples or 96-byte
# Jacobian points), tau, and the SpartanProof the prover's transcript saw.  pf.c is not used: the library derives c.
SpartanItem = Tuple[int, Sequence[int], object, object, Sequence[int], object]


def spartan_records(shape, curve: int, items: Sequence[SpartanItem]) -> Tuple[bytes, bytes, bytes, bytes]:
    """The four proof-major records vdfgpu_spartan_verify_batch reads (include/vdfgpu.h): (u, X), (comm_W, comm_E,
    L_j, R_j), the prover's scalars and the transcript's challenges, as bytes.  A commitment None is the identity."""
    from .encoding import CURVE_BASE
    from .nova import _point_arg
    m = shape.m
    base = CURVE_BASE[curve]
    inst, pts, proof, chal = [], [], [], []
    point = lambda c: bytes(96) if c is None else _point_arg(c, base)   # noqa: E731  (None: the identity)
    for u, X, comm_W, comm_E, tau, pf in items:
        if len(X) != shape.num_io:
            raise ValueError("spartan_verify_batch: X needs num_io entries")
        inst.append(fes_to_bytes([u] + list(X), m))
        pts.append(point(comm_W) + point(comm_E) + b"".join(L for L, _, _ in pf.ipa) +
                   b"".join(R for _, R, _ in pf.ipa))
        proof.append(fes_to_bytes([v for e, _ in pf.outer for v in e] + list(pf.outer_claims) +
                                  [v for e, _ in pf.inner for v in e] + list(pf.eval_claims) + [pf.a_hat], m))
        chal.append(fes_to_bytes(list(tau) + pf.r_x + list(pf.r_abc) + pf.r_y + [pf.rho, pf.u_scale] +
                                 [r for _, _, r in pf.ipa], m))
    return b"".join(inst), b"".join(pts), b"".join(proof), b"".join(chal)


def spartan_verify_records(shape, ipa_gens, k: int, inst: bytes, pts: bytes, proof: bytes, chal: bytes,
                           weights: Sequence[int] | None = None) -> List[bool]:
    """vdfgpu_spartan_verify_batch on records already encoded (spartan_records); weights as in spartan_verify_batch."""
    import secrets
    m = shape.m
    if weights is None:
        weights = [1 + secrets.randbelow(m - 1) for _ in range(k)]
    if len(weights) != k:
        raise ValueError("spartan_verify_batch: one weight per proof")
    ok = bytearray(max(k, 1))
    _lib.check(_lib.load().vdfgpu_spartan_verify_batch(shape._h, ipa_gens._h, k, _lib.as_ptr(inst), _lib.as_ptr(pts),
                                                       _lib.as_ptr(proof), _lib.as_ptr(chal),
                                                       _lib.as_ptr(fes_to_bytes(weights, m) or bytes(32)),
                                                       _lib.as_ptr(ok)))
    return [bool(v) for v in ok[:k]]


def spartan_verify_batch(shape, ipa_gens, items: Sequence[SpartanItem], weights: Sequence[int] | None = None) -> List[bool]:
    """RelaxedR1CSSNARK::verify [R] of k proofs over one shape (nova.R1CSShape) in one call, one verdict per proof.
    ipa_gens: at least m + 1 points of the curve whose scalar field is the shape's (U0 = G_m).  Every proof's
    challenges must be what the caller's transcript derived from it.  weights: one non-zero weight per proof for the
    random linear combination of the openings; None draws them with `secrets`.  A caller that passes its own must draw
    them uniformly and out of the provers' sight: predictable weights let two invalid openings cancel."""
    if not items:
        return []
    inst, pts, proof, chal = spartan_records(shape, ipa_gens.curve, items)
    return spartan_verify_records(shape, ipa_gens, len(items), inst, pts, proof, chal, weights)
