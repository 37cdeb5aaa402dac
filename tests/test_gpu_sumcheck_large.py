"""GPU: the sum-check reductions (sumcheck.cuh) at the sizes where their multi-block paths run -- grid-stride loops of
more than one iteration (2^(ell-1) > 148 * 8 * 256 items, ell >= 20), more than 256 block partials in the final kernel
(ell >= 18) -- up to the benchmark's 2^24-entry tables, against exact references:

  * tensor-product tables A = eq(a), B = eq(b), C = eq(c), D = eq(d): after binding the top k variables every table is
    a scalar times an eq table of the rest, so every round's (e0, e2, e3), the claim and the final evaluations have
    O(ell) closed forms (checked against the oracle's sum-check on the CPU below);
  * random tables against the oracle's sum-check at Nova's sizes (2^17, 2^18);
  * inner products and linear combinations at lengths around the block and grid sizes;
  * points_lincomb with outputs at infinity inside one 4-output chunk;
  * both Spartan phases at t = 1024 on the IO-bound step instance (X read by constraints)."""
import ctypes
import random

import pytest

from oracle import pasta as O
from tests import shape_gen as S
from vdf_b200 import _lib
from vdf_b200 import spartan as SP

gpu = pytest.mark.gpu


def _challenge(m, salt):
    return lambda rnd, evals: (sum(evals) * 0x9E3779B97F4A7C15 + rnd + salt) % m


# ---- closed forms over eq tables ---------------------------------------------------------------------------------
def _f(x, t, m):
    """factor of one variable of eq(x) at the point t: (1 - t)(1 - x) + t x"""
    return ((1 - t) * (1 - x) + t * x) % m


def eq_closed_form(vecs, rs, m):
    """(per-round evaluations, claim, final evaluations) of the sum-check over the tables eq(v) for v in vecs with
    challenges rs: cubic with comb = A (B C - D) for four vectors, quadratic with comb = A B for two."""
    ell = len(vecs[0])
    cubic = len(vecs) == 4
    terms = [((0, 1, 2), 1), ((0, 3), m - 1)] if cubic else [((0, 1), 1)]
    points = (0, 2, 3) if cubic else (0, 2)

    def prod_f(g, j, t):
        p = 1
        for i in g:
            p = p * _f(vecs[i][j], t, m) % m
        return p

    def bit_sum(g, j):   # sum over the variable's two values of the product of the factors
        p0 = p1 = 1
        for i in g:
            p0, p1 = p0 * (1 - vecs[i][j]) % m, p1 * vecs[i][j] % m
        return (p0 + p1) % m

    suffix = {}
    for g, _ in terms:
        s = [1] * (ell + 1)
        for j in reversed(range(ell)):
            s[j] = s[j + 1] * bit_sum(g, j) % m
        suffix[g] = s
    pref = {g: 1 for g, _ in terms}
    rounds = []
    for k in range(ell):
        rounds.append(tuple(sum(sign * pref[g] * prod_f(g, k, t) * suffix[g][k + 1] for g, sign in terms) % m
                            for t in points))
        for g, _ in terms:
            pref[g] = pref[g] * prod_f(g, k, rs[k]) % m
    claim = sum(sign * suffix[g][0] for g, sign in terms) % m
    final = []
    for v in vecs:
        p = 1
        for j in range(ell):
            p = p * _f(v[j], rs[j], m) % m
        final.append(p)
    return rounds, claim, final


def eq_entry(v, idx, m):
    ell = len(v)
    p = 1
    for j in range(ell):
        p = p * (v[j] if (idx >> (ell - 1 - j)) & 1 else 1 - v[j]) % m
    return p


@pytest.mark.parametrize("ntab", [4, 2])
def test_closed_forms_match_the_oracle(ntab):
    """CPU: the closed forms above against O.sumcheck_prove on explicit eq tables (pins the reference)."""
    m = O.Q
    py = random.Random(ntab)
    ell = 7
    vecs = [[py.randrange(m) for _ in range(ell)] for _ in range(ntab)]
    evals, rs, fin = O.sumcheck_prove([O.eq_evals(v, m) for v in vecs], m, _challenge(m, 5))
    rounds, claim, final = eq_closed_form(vecs, rs, m)
    assert [tuple(e) for e in evals] == rounds and fin == final
    tabs = [O.eq_evals(v, m) for v in vecs]
    want = sum(a * (b * c - d) for a, b, c, d in zip(*tabs)) if ntab == 4 else sum(a * b for a, b in zip(*tabs))
    assert claim == want % m
    assert all(eq_entry(vecs[0], i, m) == tabs[0][i] for i in range(1 << ell))


# ---- device helpers -------------------------------------------------------------------------------------------
def _sync_torch():
    import torch
    torch.cuda.synchronize()


def _eq_dev(lib, fid, v):
    import torch
    t = torch.empty(32 << len(v), dtype=torch.uint8, device="cuda")
    _sync_torch()
    _lib.check(lib.vdfgpu_eq_evals_dev(fid, _lib.as_ptr(O.fes_to_bytes(v, O.MODULUS[fid])), len(v), t.data_ptr()))
    _lib.check(lib.vdfgpu_synchronize())
    return t


def _entries(t, idx, m):
    import torch
    rows = t.view(-1, 32)[torch.tensor(idx, device=t.device)].cpu().numpy().tobytes()
    return O.fes_from_bytes(rows, m)


def _sumcheck_dev(lib, fid, tabs, challenge):
    m = O.MODULUS[fid]
    ell = (tabs[0].numel() // 32).bit_length() - 1
    log: list = []
    cb = SP._round_trampoline(m, challenge, log)
    final = bytearray(32 * len(tabs))
    _sync_torch()
    fn = lib.vdfgpu_sumcheck_cubic_dev if len(tabs) == 4 else lib.vdfgpu_sumcheck_quad_dev
    _lib.check(fn(fid, *[t.data_ptr() for t in tabs], ell, ctypes.cast(cb, ctypes.c_void_p), None, _lib.as_ptr(final)))
    return [e for e, _ in log], [r for _, r in log], O.fes_from_bytes(bytes(final), m)


def _poly_evaluate_dev(lib, fid, t, r):
    m = O.MODULUS[fid]
    out = bytearray(32)
    _sync_torch()
    _lib.check(lib.vdfgpu_poly_evaluate_dev(fid, t.data_ptr(), _lib.as_ptr(O.fes_to_bytes(r, m)), len(r), _lib.as_ptr(out)))
    return O.fe_from_bytes(bytes(out), m)


def _inner_product_of_dev(lib, fid, a, b):
    """vdfgpu_inner_product (host arrays) over two device tables brought back to the host"""
    ah, bh = a.cpu().numpy(), b.cpu().numpy()
    out = bytearray(32)
    _lib.check(lib.vdfgpu_inner_product(fid, ah.ctypes.data, bh.ctypes.data, a.numel() // 32, _lib.as_ptr(out)))
    return O.fe_from_bytes(bytes(out), O.MODULUS[fid])


def _ip_eq(a, b, m):
    p = 1
    for x, y in zip(a, b):
        p = p * (x * y + (1 - x) * (1 - y)) % m
    return p


@gpu
@pytest.mark.parametrize("fid,ell", [(O.FIELD_FQ, 18), (O.FIELD_FP, 20), (O.FIELD_FQ, 24)])
def test_eq_tables_sumcheck_at_large_sizes(gpu_lib, fid, ell):
    """eq_evals_dev, poly_evaluate_dev, inner_product and the cubic and quadratic sum-checks on 2^ell-entry eq tables,
    every round compared exactly with the closed form.  ell = 24 is the benchmark's size (4 x 512 MiB)."""
    lib = gpu_lib
    m = O.MODULUS[fid]
    py = random.Random(ell * 10 + fid)
    vecs = [[py.randrange(m) for _ in range(ell)] for _ in range(4)]
    vecs[1][0], vecs[2][ell - 1] = 0, 1          # boolean coordinates: half of a table is zero
    tabs = [_eq_dev(lib, fid, v) for v in vecs]
    n = 1 << ell
    idx = sorted({0, 1, n - 2, n - 1, n // 2, n // 2 - 1} | {py.randrange(n) for _ in range(300)})
    for v, t in zip(vecs, tabs):
        assert _entries(t, idx, m) == [eq_entry(v, i, m) for i in idx]
    assert _poly_evaluate_dev(lib, fid, tabs[0], vecs[3]) == _ip_eq(vecs[0], vecs[3], m)
    assert _inner_product_of_dev(lib, fid, tabs[2], tabs[3]) == _ip_eq(vecs[2], vecs[3], m)
    quad = [t.clone() for t in tabs[:2]]
    evals, rs, fin = _sumcheck_dev(lib, fid, tabs, _challenge(m, ell))
    rounds, claim, final = eq_closed_form(vecs, rs, m)
    assert len(evals) == ell and evals == rounds and fin == final
    assert _verify_rounds(claim, evals, rs, m, cubic=True) == fin[0] * (fin[1] * fin[2] - fin[3]) % m
    del tabs
    evals, rs, fin = _sumcheck_dev(lib, fid, quad, _challenge(m, ell + 1))
    rounds, _, final = eq_closed_form(vecs[:2], rs, m)
    assert evals == rounds and fin == final


@gpu
@pytest.mark.parametrize("fid,ell", [(O.FIELD_FQ, 18), (O.FIELD_FP, 17)])
def test_random_tables_against_the_oracle(gpu_lib, fid, ell):
    """Nova's own table sizes: host-table and device-table forms of both sum-checks against O.sumcheck_prove."""
    import torch
    lib = gpu_lib
    m = O.MODULUS[fid]
    py = random.Random(ell + 100 * fid)
    tabs = [[py.randrange(m) for _ in range(1 << ell)] for _ in range(4)]
    tabs[0][5], tabs[1][(1 << ell) - 1], tabs[3][1 << (ell - 1)] = 0, m - 1, 1
    for k in (4, 2):
        ch = _challenge(m, 7 * k)
        want = O.sumcheck_prove(tabs[:k], m, ch)
        got = SP.sumcheck(fid, tabs[:k], ch)
        assert got[0] == [tuple(e) for e in want[0]] and got[1] == want[1] and got[2] == want[2]
        dev = [torch.frombuffer(bytearray(O.fes_to_bytes(t, m)), dtype=torch.uint8).cuda() for t in tabs[:k]]
        assert _sumcheck_dev(lib, fid, dev, ch) == got


@gpu
@pytest.mark.parametrize("fid", [O.FIELD_FP, O.FIELD_FQ])
def test_eq_evals_and_poly_evaluate_up_to_16(gpu_lib, fid):
    import torch
    lib = gpu_lib
    m = O.MODULUS[fid]
    py = random.Random(30 + fid)
    for ell in (12, 13, 15, 16):
        r = [py.randrange(m) for _ in range(ell)]
        want = O.eq_evals(r, m)
        assert SP.eq_evals(fid, r) == want
        t = _eq_dev(lib, fid, r)
        assert O.fes_from_bytes(t.cpu().numpy().tobytes(), m) == want
        poly = [py.randrange(m) for _ in range(1 << ell)]
        pv = O.poly_evaluate(poly, r, m)
        assert SP.poly_evaluate(fid, poly, r) == pv
        pd = torch.frombuffer(bytearray(O.fes_to_bytes(poly, m)), dtype=torch.uint8).cuda()
        assert _poly_evaluate_dev(lib, fid, pd, r) == pv


@gpu
@pytest.mark.parametrize("n", [1, 255, 256, 257, 65537, 303104, 303105, (1 << 20) + 3])
def test_inner_product_and_vec_lincomb_lengths(gpu_lib, n):
    """Around one block (256), one full grid pass (148 * 8 * 256 = 303104) and beyond."""
    fid = O.FIELD_FQ if n % 2 else O.FIELD_FP
    m = O.MODULUS[fid]
    py = random.Random(n)
    a, b = S.random_vec(py, m, n), S.random_vec(py, m, n)
    a[-1], b[-1] = m - 1, m - 1          # the last element must be summed too
    assert SP.inner_product(fid, a, b) == sum(x * y for x, y in zip(a, b)) % m
    x, y = py.randrange(m), m - 1
    assert SP.vec_lincomb(fid, a, b, x, y) == [(x * p + y * q) % m for p, q in zip(a, b)]


@gpu
@pytest.mark.parametrize("cid", [O.CURVE_PALLAS, O.CURVE_VESTA])
def test_points_lincomb_infinity_inside_a_chunk(gpu_lib, cid):
    """Outputs at infinity between finite outputs of one 4-output chunk (the batched inversion skips them), lengths
    n = 1, 2, 3 (mod 4), weights 0, 1 and order - 1.  Q = kP with k random, k = 1 (the precomputed P + Q doubles) and
    k = -1 (P + Q is the identity); one P given as the identity with the x / y bytes of a real point, which the
    infinity flag overrides."""
    cv = O.CURVES[cid]
    m = cv.order
    py = random.Random(70 + cid)
    for n in (9, 14, 23):
        P = [cv.mul(py.randrange(1, m), cv.gen) for _ in range(n)]
        junk = O.affine_to_bytes(cv, P[n - 3])[:64] + b"\x01" + bytes(7)
        P[n - 3] = None
        Pb = O.affines_to_bytes(cv, P[:n - 3]) + junk + O.affines_to_bytes(cv, P[n - 2:])
        for k in (py.randrange(2, m), 1, m - 1):
            Q = [cv.mul(py.randrange(1, m), cv.gen) for _ in range(n)]
            for i in range(1, n, 4):          # Q = k P at positions 1, 5, 9, ...: w1 P + w2 Q = (w1 + k w2) P
                Q[i] = cv.mul(k, P[i])
            Q[n - 1] = cv.mul(k, P[n - 1])    # and the last output of the ragged last chunk
            for w2 in (py.randrange(1, m), 1, m - 1):
                w1 = (-k * w2) % m
                got = SP.points_lincomb(cid, Pb, O.affines_to_bytes(cv, Q), w1, w2)
                want = [cv.add(cv.mul(w1, p), cv.mul(w2, q)) for p, q in zip(P, Q)]
                assert want[1] is None and want[0] is not None and want[2] is not None
                assert [O.affine_from_bytes(cv, got[72 * i:72 * i + 72]) for i in range(n)] == want, (n, k, w2)
            for w1, w2 in ((0, 1), (1, 0), (m - 1, 1), (0, 0)):
                got = SP.points_lincomb(cid, Pb, O.affines_to_bytes(cv, Q), w1, w2)
                want = [cv.add(cv.mul(w1, p), cv.mul(w2, q)) for p, q in zip(P, Q)]
                assert [O.affine_from_bytes(cv, got[72 * i:72 * i + 72]) for i in range(n)] == want, (n, k, w1, w2)


def _interp(points, r, m):
    acc = 0
    for k, (xk, yk) in enumerate(points):
        num, den = 1, 1
        for j, (xj, _) in enumerate(points):
            if j != k:
                num, den = num * (r - xj) % m, den * (xk - xj) % m
        acc = (acc + yk * num * pow(den, -1, m)) % m
    return acc


def _verify_rounds(claim, evals, rs, m, cubic):
    for e, r in zip(evals, rs):
        pts = [(0, e[0]), (1, (claim - e[0]) % m), (2, e[1])] + ([(3, e[2])] if cubic else [])
        claim = _interp(pts, r, m)
    return claim


@gpu
def test_spartan_phases_at_t1024_on_the_io_bound_shape(gpu_lib):
    """test_gpu_sumcheck.py's two Spartan phases on a folded relaxed instance of the IO-bound step shape at t = 1024
    with the 9800-constraint augmented block: z and bind_rows' output have non-zero X parts."""
    from vdf_b200 import nova as N
    fid, m = O.FIELD_FQ, O.Q
    py = random.Random(1024)
    shape, W1, X1 = S.fresh_instance(fid, 1024, 0, 9800)
    _, W2, X2 = S.fresh_instance(fid, 1024, 1, 9800)
    r_fold = py.randrange(1 << 128)
    T = shape.cross_term(W1, 1, X1, W2, X2)
    W, E = O.fold_vec(W1, W2, r_fold, m), [r_fold * t % m for t in T]
    X, u = O.fold_vec(X1, X2, r_fold, m), (1 + r_fold) % m
    assert shape.is_sat_relaxed(W, E, u, X) and any(E)
    z = shape.z_of(W, u, X)
    gs = N.R1CSShape(fid, shape.num_cons, shape.num_vars, shape.num_io, shape.A, shape.B, shape.C)
    Az, Bz, Cz = gs.multiply_vec(z)

    def pad(v, ell):
        return list(v) + [0] * ((1 << ell) - len(v))

    ch = _challenge(m, 999)
    ell_x = max(1, (shape.num_cons - 1).bit_length())
    tau = [py.randrange(m) for _ in range(ell_x)]
    D = [(u * c + e) % m for c, e in zip(Cz, E)]
    evals, rx, fin = SP.sumcheck(fid, [SP.eq_evals(fid, tau), pad(Az, ell_x), pad(Bz, ell_x), pad(D, ell_x)], ch)
    assert _verify_rounds(0, evals, rx, m, cubic=True) == fin[0] * (fin[1] * fin[2] - fin[3]) % m
    assert fin[0] == O.poly_evaluate(O.eq_evals(tau, m), rx, m)
    claim_Cz = SP.poly_evaluate(fid, pad(Cz, ell_x), rx)
    assert fin[3] == (u * claim_Cz + SP.poly_evaluate(fid, pad(E, ell_x), rx)) % m
    r_abc = [py.randrange(m) for _ in range(3)]
    eq_rx = SP.eq_evals(fid, rx)[:shape.num_cons]
    Mt = gs.bind_rows(eq_rx, r_abc)
    assert Mt == shape.bind_rows(eq_rx, r_abc)
    nv = shape.num_vars
    assert all(Mt[nv + 1:]) and all(z[nv + 1:])
    ell_y = max(1, (len(z) - 1).bit_length())
    claim = (r_abc[0] * fin[1] + r_abc[1] * fin[2] + r_abc[2] * claim_Cz) % m
    evals, ry, fin2 = SP.sumcheck(fid, [pad(Mt, ell_y), pad(z, ell_y)], ch)
    assert _verify_rounds(claim, evals, ry, m, cubic=False) == fin2[0] * fin2[1] % m
    eq_ry, eq_rx_full = O.eq_evals(ry, m), O.eq_evals(rx, m)
    want = 0
    for M, rm in zip((shape.A, shape.B, shape.C), r_abc):
        want = (want + rm * sum(v * eq_rx_full[r] % m * eq_ry[c] for r, c, v in M)) % m
    assert fin2[0] == want
    assert fin2[1] == O.poly_evaluate(pad(z, ell_y), ry, m)
    gs.close()
