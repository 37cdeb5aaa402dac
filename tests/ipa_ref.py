"""The inner-product argument of spartan_with_ipa_pc [R] restated with Python integers on oracle/pasta.py curves: the
prover with folded generators, the verifier, the tables the device computes instead of folding (coef_j, the
commitment scalars SL / SR, s), and a known-discrete-log tracker for generator sets P_i = (k0 + i d) G.
Notation as in vdf_b200/csrc/sumcheck.cuh: n = 2^ell, G_n = U0, U = u_scale U0."""
from typing import Callable, List, Sequence

from oracle import pasta as O

Challenge = Callable[[int, bytes, bytes], int]


def inner(a: Sequence[int], b: Sequence[int], m: int) -> int:
    return sum(x * y for x, y in zip(a, b)) % m


def coef_next(coef: Sequence[int], r: int, m: int) -> List[int]:
    """coef_{j+1}[2t + beta] = coef_j[t] (beta ? r : r^-1)"""
    ri = pow(r, -1, m)
    return [c * f % m for c in coef for f in (ri, r)]


def coef_tables(rs: Sequence[int], m: int) -> List[List[int]]:
    """[coef_0, ..., coef_ell]"""
    out = [[1]]
    for r in rs:
        out.append(coef_next(out[-1], r, m))
    return out


def s_table(rs: Sequence[int], m: int) -> List[int]:
    """s_k = prod_j (bit_j(k) ? r_j : r_j^-1), bit_0 the most significant of the ell bits, straight from the
    definition (independent of coef_next)."""
    ell = len(rs)
    inv = [pow(r, -1, m) for r in rs]
    out = []
    for k in range(1 << ell):
        v = 1
        for j in range(ell):
            v = v * (rs[j] if (k >> (ell - 1 - j)) & 1 else inv[j]) % m
        out.append(v)
    return out


def expand(a: Sequence[int], coef: Sequence[int], n: int, cL: int, cR: int, u_scale: int, m: int):
    """The scalars of L and R over G[0, n] for the current a (length mm = n / len(coef)): k = t mm + i."""
    mm = len(a)
    h = mm // 2
    SL, SR = [0] * (n + 1), [0] * (n + 1)
    for k in range(n):
        t, i = divmod(k, mm)
        if i >= h:
            SL[k] = a[i - h] * coef[t] % m
        else:
            SR[k] = a[i + h] * coef[t] % m
    SL[n], SR[n] = cL * u_scale % m, cR * u_scale % m
    return SL, SR


def fold(a: Sequence[int], b: Sequence[int], r: int, m: int):
    h = len(a) // 2
    ri = pow(r, -1, m)
    return ([(r * x + ri * y) % m for x, y in zip(a[:h], a[h:])],
            [(ri * x + r * y) % m for x, y in zip(b[:h], b[h:])])


def prove(cv: O.Curve, G: Sequence, U0, u_scale: int, a: Sequence[int], b: Sequence[int], challenge: Challenge):
    """The round loop with folded generators.  Returns (L list, R list, challenges, a_hat), points as affine tuples;
    the challenge sees them as the library hands them over (96-byte normalised)."""
    m = cv.order
    U = cv.mul(u_scale, U0)
    a, b, G = list(a), list(b), list(G)
    Ls, Rs, rs = [], [], []
    rnd = 0
    while len(a) > 1:
        h = len(a) // 2
        cL, cR = inner(a[:h], b[h:], m), inner(a[h:], b[:h], m)
        L = cv.add(cv.msm_naive(a[:h], G[h:]), cv.mul(cL, U))
        R = cv.add(cv.msm_naive(a[h:], G[:h]), cv.mul(cR, U))
        r = challenge(rnd, O.jac_to_bytes(cv, L), O.jac_to_bytes(cv, R)) % m
        ri = pow(r, -1, m)
        a, b = fold(a, b, r, m)
        G = [cv.add(cv.mul(ri, x), cv.mul(r, y)) for x, y in zip(G[:h], G[h:])]
        Ls.append(L)
        Rs.append(R)
        rs.append(r)
        rnd += 1
    return Ls, Rs, rs, a[0]


def verify(cv: O.Curve, G: Sequence, U0, u_scale: int, P, b: Sequence[int], Ls, Rs, rs, a_hat: int) -> bool:
    """P' = r^2 L + P + r^-2 R per round, then P_final == a_hat (G_hat + b_hat U) with G_hat = <s, G>, b_hat = <b, s>.
    P = commit(a) + <a, b> U."""
    m = cv.order
    U = cv.mul(u_scale, U0)
    for L, R, r in zip(Ls, Rs, rs):
        ri = pow(r, -1, m)
        P = cv.add(cv.add(cv.mul(r * r, L), P), cv.mul(ri * ri, R))
    s = s_table(rs, m)
    G_hat = cv.msm_naive(s, G)
    b_hat = inner(b, s, m)
    return P == cv.mul(a_hat, cv.add(G_hat, cv.mul(b_hat, U)))


class DlogTracker:
    """The prover's rounds on the discrete logs of G_i = (k0 + i d) G (and U0 = G_n) instead of the points: the logs
    of L_j and R_j for the library's challenges in O(n) integer operations per round.  point(log) is one cv.mul."""

    def __init__(self, cv: O.Curve, k0: int, d: int, ell: int, u_scale: int, a: Sequence[int], b: Sequence[int]):
        self.cv, self.m = cv, cv.order
        n = 1 << ell
        self.g = [(k0 + i * d) % self.m for i in range(n)]
        self.u = (k0 + n * d) * u_scale % self.m
        self.a, self.b = list(a), list(b)

    def point(self, log: int):
        return self.cv.mul(log % self.m, self.cv.gen)

    def round(self, r: int):
        """(log L, log R) of the current round, then the fold with r."""
        m, a, b, g = self.m, self.a, self.b, self.g
        h = len(a) // 2
        cL, cR = inner(a[:h], b[h:], m), inner(a[h:], b[:h], m)
        logL = (inner(a[:h], g[h:], m) + cL * self.u) % m
        logR = (inner(a[h:], g[:h], m) + cR * self.u) % m
        ri = pow(r, -1, m)
        self.a, self.b = fold(a, b, r, m)
        self.g = [(ri * x + r * y) % m for x, y in zip(g[:h], g[h:])]
        return logL, logR
