"""RelaxedR1CSSNARK::prove and ::verify of nova-snark 0.8 spartan_with_ipa_pc [R] restated with Python integers on
nova's padded layout, driven by the same transcript object as nova.RunningProver.spartan_prove (sumcheck_round,
claims, ipa_round): the test oracle of vdfgpu_running_spartan_prove and vdfgpu_r1cs_evaluate.  The padding is restated
here on purpose, independently of the library and of vdf_b200.spartan.padded_layout.  Notation as in
vdf_b200/csrc/sumcheck.cuh."""
import hashlib
from typing import List, Sequence, Tuple

from oracle import pasta as O
from tests import ipa_ref as IR
from vdf_b200.nova import SpartanProof


class Transcript:
    """deterministic stand-in for nova's transcript: every answer a hash of the stage and what it was handed"""

    def __init__(self, salt: int = 0):
        self.salt = salt

    def _h(self, *xs):
        return int.from_bytes(hashlib.sha256(repr((self.salt,) + xs).encode()).digest(), "little")

    def sumcheck_round(self, rnd, evals):
        return self._h("round", rnd, evals)

    def claims(self, stage, values):
        return [self._h("claims", stage, values, k) for k in range((3, 1, 1)[stage])]

    def ipa_round(self, rnd, L, R):
        return self._h("ipa", rnd, L, R)


def padded_size(shape: O.R1CSShape) -> int:
    """m: the smallest power of two that holds both the constraints and the witness variables"""
    m = 1
    while m < shape.num_cons or m < shape.num_vars:
        m *= 2
    return m


def padded_entries(shape: O.R1CSShape) -> List[List[Tuple[int, int, int]]]:
    """A, B, C with u and X moved to columns m, m + 1, ... (W keeps columns 0 .. num_vars - 1)"""
    shift = padded_size(shape) - shape.num_vars
    return [[(r, c if c < shape.num_vars else c + shift, v) for r, c, v in M] for M in (shape.A, shape.B, shape.C)]


def padded_z(shape: O.R1CSShape, W: Sequence[int], u: int, X: Sequence[int]) -> List[int]:
    m = padded_size(shape)
    return list(W) + [0] * (m - len(W)) + [u] + list(X) + [0] * (m - 1 - len(X))


def evaluate(shape: O.R1CSShape, rx: Sequence[int], ry: Sequence[int]) -> Tuple[int, int, int]:
    """(A, B, C)(r_x, r_y) straight from the padded entries"""
    p = shape.m
    ex, ey = O.eq_evals(rx, p), O.eq_evals(ry, p)
    return tuple(sum(v * ex[r] % p * ey[c] for r, c, v in M) % p for M in padded_entries(shape))


def _pad(v: Sequence[int], n: int) -> List[int]:
    return list(v) + [0] * (n - len(v))


def prove(shape: O.R1CSShape, W, E, u: int, X, tau: Sequence[int], transcript, cv: O.Curve, G: Sequence) -> SpartanProof:
    """The prover over the running instance (W, E, u, X); G: the IPA set as affine points (m + 1 of them, U0 = G[m])."""
    p = shape.m
    m = padded_size(shape)
    assert 1 + shape.num_io <= m and len(tau) == m.bit_length() - 1
    Wp, Ep = _pad(W, m), _pad(E, m)
    Az, Bz, Cz = (_pad(v, m) for v in shape.multiply_vec(shape.z_of(W, u, X)))
    D = [(u * c + e) % p for c, e in zip(Cz, Ep)]

    def sc(rnd, evals):
        return transcript.sumcheck_round(rnd, tuple(evals)) % p

    def claims(stage, vals):
        return tuple(v % p for v in transcript.claims(stage, tuple(vals)))

    outer_evals, rx, fin = O.sumcheck_prove([O.eq_evals(tau, p), Az, Bz, D], p, sc)
    eq_rx = O.eq_evals(rx, p)
    outer_claims = (fin[1], fin[2], IR.inner(Cz, eq_rx, p), IR.inner(Ep, eq_rx, p))
    r_abc = claims(0, outer_claims)
    Mp = [0] * (2 * m)
    for M, rm in zip(padded_entries(shape), r_abc):
        for r, c, v in M:
            Mp[c] = (Mp[c] + rm * v % p * eq_rx[r]) % p
    inner_evals, ry, _ = O.sumcheck_prove([Mp, padded_z(shape, W, u, X)], p, sc)
    eq_ry = O.eq_evals(ry[1:], p)
    eval_W = IR.inner(Wp, eq_ry, p)
    T = (IR.inner(Ep, eq_ry, p) + IR.inner(Wp, eq_rx, p)) % p
    (rho,) = claims(1, (eval_W, T))
    a = [(e + rho * w) % p for e, w in zip(Ep, Wp)]
    b = [(x + rho * y) % p for x, y in zip(eq_rx, eq_ry)]
    c = (outer_claims[3] + rho * T + rho * rho * eval_W) % p
    assert c == IR.inner(a, b, p)
    (u_scale,) = claims(2, (c,))
    Ls, Rs, rs, a_hat = IR.prove(cv, G[:m], G[m], u_scale, a, b, transcript.ipa_round)
    return SpartanProof(list(zip(outer_evals, rx)), outer_claims, r_abc, list(zip(inner_evals, ry)), (eval_W, T), rho,
                        c, u_scale, [(O.jac_to_bytes(cv, L), O.jac_to_bytes(cv, R), r) for L, R, r in zip(Ls, Rs, rs)],
                        a_hat)


def _interp(points, r: int, p: int) -> int:
    acc = 0
    for k, (xk, yk) in enumerate(points):
        num, den = 1, 1
        for j, (xj, _) in enumerate(points):
            if j != k:
                num = num * (r - xj) % p
                den = den * (xk - xj) % p
        acc = (acc + yk * num * pow(den, -1, p)) % p
    return acc


def _rounds(claim: int, rounds, p: int) -> int:
    """the sum-check verifier, O(ell): e(0) + e(1) = claim, the next claim is e(r)"""
    for e, r in rounds:
        pts = [(0, e[0]), (1, (claim - e[0]) % p)] + [(k + 2, v) for k, v in enumerate(e[1:])]
        claim = _interp(pts, r, p)
    return claim


def verify_claims(shape: O.R1CSShape, u: int, X: Sequence[int], tau: Sequence[int], pf: SpartanProof,
                  abc=None) -> bool:
    """Everything of RelaxedR1CSSNARK::verify except the opening and the transcript: both sum-checks round by round,
    their final claims (abc = (A, B, C)(r_x, r_y), computed here when None; z(r_y) from eval_W and the public [u, X]),
    and the joint claim c.  The opening is the inner-product claim <E + rho W, eq(r_x) + rho eq(r_y')> = c under
    comm_E + rho comm_W."""
    p = shape.m
    m = padded_size(shape)
    rx, ry = pf.r_x, pf.r_y
    if len(rx) != m.bit_length() - 1 or len(ry) != len(rx) + 1:
        return False
    cAz, cBz, cCz, eval_E = pf.outer_claims
    if _rounds(0, pf.outer, p) != O.poly_evaluate(O.eq_evals(tau, p), rx, p) * (cAz * cBz - u * cCz - eval_E) % p:
        return False
    rA, rB, rC = pf.r_abc
    A, B, C = evaluate(shape, rx, ry) if abc is None else abc
    eval_W, T = pf.eval_claims
    eval_X = O.poly_evaluate(_pad([u] + list(X), m), ry[1:], p)
    z_ry = ((1 - ry[0]) * eval_W + ry[0] * eval_X) % p
    if _rounds((rA * cAz + rB * cBz + rC * cCz) % p, pf.inner, p) != (rA * A + rB * B + rC * C) * z_ry % p:
        return False
    return pf.c == (eval_E + pf.rho * T + pf.rho * pf.rho * eval_W) % p


def transcript_consistent(pf: SpartanProof, transcript, p: int) -> bool:
    """every challenge and answer of the proof is what the transcript derives from what it was handed"""
    for rounds in (pf.outer, pf.inner):
        if any(r != transcript.sumcheck_round(j, tuple(e)) % p for j, (e, r) in enumerate(rounds)):
            return False
    stages = ((0, pf.outer_claims, pf.r_abc), (1, pf.eval_claims, (pf.rho,)), (2, (pf.c,), (pf.u_scale,)))
    if any(tuple(v % p for v in transcript.claims(s, tuple(i))) != tuple(o) for s, i, o in stages):
        return False
    return all(r == transcript.ipa_round(j, L, R) % p for j, (L, R, r) in enumerate(pf.ipa))
