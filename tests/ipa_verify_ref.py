"""Batch verification of inner-product arguments restated with Python integers on oracle/pasta.py curves, in the
notation of vdf_b200/csrc/sumcheck.cuh: proof q is valid iff
    a_hat G_hat + u_scale (a_hat b_hat - c) U0 - comm_a - sum_j (r_j^2 L_j + r_j^-2 R_j) = O,   G_hat = <s, G[0,n)>,
and a batch with weights w_q passes iff the weighted sum of the k left-hand sides is O.  A proof here is
(Ls, Rs, rs, a_hat, comm_a, c, b_hat, u_scale) with points as affine tuples (None = identity)."""
from typing import List, Sequence

from oracle import pasta as O
from tests import ipa_ref as IR


def lhs(cv: O.Curve, G: Sequence, U0, proof):
    """The left-hand side of proof q's equation (None = O)."""
    Ls, Rs, rs, a_hat, comm_a, c, b_hat, u_scale = proof
    m = cv.order
    acc = cv.msm_naive([a_hat * s % m for s in IR.s_table(rs, m)], G)
    acc = cv.add(acc, cv.mul(u_scale * (a_hat * b_hat - c) % m, U0))
    acc = cv.add(acc, cv.neg(comm_a))
    for L, R, r in zip(Ls, Rs, rs):
        ri = pow(r, -1, m)
        acc = cv.add(acc, cv.neg(cv.add(cv.mul(r * r, L), cv.mul(ri * ri, R))))
    return acc


def verify_one(cv: O.Curve, G: Sequence, U0, proof) -> bool:
    return lhs(cv, G, U0, proof) is None


def batch_passes(cv: O.Curve, G: Sequence, U0, proofs, weights: Sequence[int]) -> bool:
    acc = None
    for p, w in zip(proofs, weights):
        acc = cv.add(acc, cv.mul(w, lhs(cv, G, U0, p)))
    return acc is None


def batch_scalars(rs_list: Sequence[Sequence[int]], scales: Sequence[int], m: int) -> List[int]:
    """S[i] = sum_q scale_q s_q[i] (i < n): the scalars of the MSM over G[0, n) (slot n is the caller's sum)."""
    n = 1 << len(rs_list[0])
    S = [0] * n
    for rs, sc in zip(rs_list, scales):
        for i, v in enumerate(IR.s_table(rs, m)):
            S[i] = (S[i] + sc * v) % m
    return S


def half_tables(rs: Sequence[int], scale: int, lo_bits: int, m: int):
    """(Hi, Lo) with s[t 2^lo_bits + u] = Hi[t] Lo[u] / scale: Hi over the first ell - lo_bits challenges (times
    scale), Lo over the rest."""
    hb = len(rs) - lo_bits
    return ([scale * v % m for v in IR.s_table(rs[:hb], m)], IR.s_table(rs[hb:], m))
