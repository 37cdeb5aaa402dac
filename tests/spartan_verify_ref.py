"""RelaxedR1CSSNARK::verify of k proofs in one batch restated with Python integers: the test oracle of
vdfgpu_spartan_verify_batch.  Built from spartan_ref.verify_claims (both sum-checks and their final claims) and
ipa_verify_ref (the openings as one weighted sum, each proof alone when the sum is not O), with c and b_hat derived
from the proof as the library derives them.  An item is (u, X, comm_W, comm_E, tau, SpartanProof) with the
commitments as affine points of oracle/pasta.py (None = identity); pf.c is not used."""
import dataclasses
from typing import List, Sequence

from oracle import pasta as O
from tests import ipa_verify_ref as VR
from tests import spartan_ref as SR
from vdf_b200 import spartan as SP


def derived_c(pf, p: int) -> int:
    eval_W, T = pf.eval_claims
    return (pf.outer_claims[3] + pf.rho * T + pf.rho * pf.rho * eval_W) % p


def opening(cv: O.Curve, fid: int, item):
    """the opening of one item as ipa_verify_ref's proof tuple: comm_a = comm_E + rho comm_W, c and b_hat derived"""
    u, X, comm_W, comm_E, tau, pf = item
    rs = [r for _, _, r in pf.ipa]
    b_hat = SP.ipa_b_hat(fid, rs, [(1, pf.r_x), (pf.rho, pf.r_y[1:])])
    return ([O.jac_from_bytes(cv, L) for L, _, _ in pf.ipa], [O.jac_from_bytes(cv, R) for _, R, _ in pf.ipa], rs,
            pf.a_hat, cv.add(comm_E, cv.mul(pf.rho, comm_W)), derived_c(pf, cv.order), b_hat, pf.u_scale)


def claims_ok(shape: O.R1CSShape, item) -> bool:
    u, X, _, _, tau, pf = item
    return SR.verify_claims(shape, u, X, tau, dataclasses.replace(pf, c=derived_c(pf, shape.m)))


def verify_one(shape: O.R1CSShape, cv: O.Curve, fid: int, G: Sequence, item) -> bool:
    """one proof: its claims, then its opening over G[0, m) with U0 = G[m]"""
    m = SR.padded_size(shape)
    return claims_ok(shape, item) and VR.verify_one(cv, G[:m], G[m], opening(cv, fid, item))


def verify_batch(shape: O.R1CSShape, cv: O.Curve, fid: int, G: Sequence, items, weights: Sequence[int]) -> List[bool]:
    """the batch as the library runs it: the claims of each proof, then the admitted openings as one weighted sum;
    when that sum is not O, each admitted opening alone"""
    m = SR.padded_size(shape)
    admitted = [q for q, it in enumerate(items) if claims_ok(shape, it)]
    ops = {q: opening(cv, fid, items[q]) for q in admitted}
    verdict = [False] * len(items)
    if admitted and VR.batch_passes(cv, G[:m], G[m], [ops[q] for q in admitted], [weights[q] for q in admitted]):
        for q in admitted:
            verdict[q] = True
    else:
        for q in admitted:
            verdict[q] = VR.verify_one(cv, G[:m], G[m], ops[q])
    return verdict


def corrupt(item, what: str, cv: O.Curve, p: int):
    """the item with one value changed: `what` is one of CORRUPTIONS; p is the scalar field"""
    u, X, cW, cE, tau, pf = item
    bump = lambda v: (v + 1) % p   # noqa: E731
    rep = dataclasses.replace
    if what == "outer round":
        pf = rep(pf, outer=[((bump(pf.outer[1][0][0]),) + pf.outer[1][0][1:], pf.outer[1][1]) if j == 1 else e
                            for j, e in enumerate(pf.outer)])
    elif what == "inner round":
        pf = rep(pf, inner=[((pf.inner[2][0][0], bump(pf.inner[2][0][1])), pf.inner[2][1]) if j == 2 else e
                            for j, e in enumerate(pf.inner)])
    elif what in ("claim_Az", "claim_Cz", "eval_E"):
        j = {"claim_Az": 0, "claim_Cz": 2, "eval_E": 3}[what]
        pf = rep(pf, outer_claims=tuple(bump(v) if i == j else v for i, v in enumerate(pf.outer_claims)))
    elif what in ("eval_W", "T"):
        j = 0 if what == "eval_W" else 1
        pf = rep(pf, eval_claims=tuple(bump(v) if i == j else v for i, v in enumerate(pf.eval_claims)))
    elif what == "a_hat":
        pf = rep(pf, a_hat=bump(pf.a_hat))
    elif what == "L_j":
        L0 = O.jac_to_bytes(cv, cv.add(O.jac_from_bytes(cv, pf.ipa[0][0]), cv.gen))
        pf = rep(pf, ipa=[(L0,) + pf.ipa[0][1:]] + pf.ipa[1:])
    elif what == "comm_W":
        cW = cv.add(cW, cv.gen)
    elif what == "comm_E":
        cE = cv.add(cE, cv.gen)
    elif what == "u":
        u = bump(u)
    elif what == "X":
        X = [bump(X[0])] + list(X[1:])
    elif what == "r_y[0]":
        pf = rep(pf, inner=[(pf.inner[0][0], bump(pf.inner[0][1]))] + pf.inner[1:])
    return (u, X, cW, cE, tau, pf)


# every value a corrupted proof can differ in, one at a time (r_y[0]: the verifier's challenge differs from the
# proof's)
CORRUPTIONS = ["outer round", "inner round", "claim_Az", "claim_Cz", "eval_E", "eval_W", "T", "a_hat", "L_j", "comm_W",
               "comm_E", "u", "X", "r_y[0]"]
