"""CPU: the library's kernel functors (the very code the GPU runs, minus the PTX multiplier) executed by a
CPU loop (tests/emul) against the oracle.  Covers the host-visible logic: digit recoding, counting sort,
range-based accumulation + record levels, reduction tree, table levels, COO->CSR, cross-term, fold."""
import ctypes
import random

import numpy as np
import pytest

from oracle import pasta as O
from tests.msm_cases import families, signed_digits
from tests.util import aligned, edge_field_values, nova_like_scalars, ptr, rand_scalars

SZ = ctypes.c_size_t


def _msm(emul, cid, table, c, S, G, logm, pts, sc, is_mont=1):
    cv = O.CURVES[cid]
    n = len(pts)
    pb = aligned(O.affines_to_bytes(cv, pts))
    sb = aligned(O.fes_to_bytes(sc, cv.order) if is_mont else b"".join(s.to_bytes(32, "little") for s in sc))
    out = np.zeros(96, np.uint8)
    assert emul.emul_msm(cid, table, c, S, G, logm, ptr(pb), SZ(n), ptr(sb), is_mont, ptr(out)) == 0
    return out.tobytes()


@pytest.mark.parametrize("fid", [O.FIELD_FP, O.FIELD_FQ])
def test_field_ops(emul, fid):
    m = O.MODULUS[fid]
    rng = O.XorShiftRng()
    edge = edge_field_values(m)
    A = [a for a in edge for _ in edge] + rand_scalars(rng, m, 200)
    B = [b for _ in edge for b in edge] + rand_scalars(rng, m, 200)
    n = len(A)
    a, b, o = aligned(O.fes_to_bytes(A, m)), aligned(O.fes_to_bytes(B, m)), np.zeros(n * 32, np.uint8)
    ops = {0: lambda x, y: x * y % m, 1: lambda x, y: (x + y) % m, 2: lambda x, y: (x - y) % m,
           3: lambda x, y: x * x % m, 6: lambda x, y: (-x) % m, 7: lambda x, y: 1}
    for op, f in ops.items():
        emul.emul_field_op(fid, op, ptr(a), ptr(b), ptr(o), SZ(n))
        assert O.fes_from_bytes(o.tobytes(), m) == [f(x, y) for x, y in zip(A, B)], op
    emul.emul_field_op(fid, 4, ptr(a), ptr(b), ptr(o), SZ(40))
    assert O.fes_from_bytes(o.tobytes()[:40 * 32], m) == [pow(x, -1, m) if x else 0 for x in A[:40]]
    emul.emul_field_op(fid, 5, ptr(a), ptr(b), ptr(o), SZ(n))  # from_mont
    assert [int.from_bytes(o.tobytes()[k:k + 32], "little") for k in range(0, n * 32, 32)] == A


@pytest.mark.parametrize("cid", [O.CURVE_PALLAS, O.CURVE_VESTA])
def test_progression(emul, cid):
    cv = O.CURVES[cid]
    for k0, d, n in ((7, 3, 50), (0, 5, 20), (1, 0, 5)):
        out = np.zeros(n * 72, np.uint8)
        emul.emul_progression(cid, ptr(aligned(k0.to_bytes(32, "little"))), ptr(aligned(d.to_bytes(32, "little"))), SZ(n), ptr(out))
        got = [O.affine_from_bytes(cv, out.tobytes()[72 * i:72 * i + 72]) for i in range(n)]
        assert got == cv.progression(k0, d, n)


@pytest.mark.parametrize("cid", [O.CURVE_PALLAS, O.CURVE_VESTA])
@pytest.mark.parametrize("table", [0, 1])
def test_msm_pipeline(emul, cid, table):
    cv = O.CURVES[cid]
    rng = O.XorShiftRng()
    n = 200
    pts = cv.progression(5, 11, n)
    sc = rand_scalars(rng, cv.order, n)
    sc[0], sc[1], sc[2], sc[3] = 0, 1, cv.order - 1, 1 << 128
    pts[7] = None
    pts[9], sc[9] = pts[8], sc[8]
    pts[11], sc[11] = cv.neg(pts[10]), sc[10]
    want = O.jac_to_bytes(cv, cv.msm(sc, pts))
    # stage 6 has three paths: c <= 3 the recursive running-sum tree, 4 <= c <= 16 the bit decomposition,
    # c >= 17 the hybrid (one running-sum level, then bit decomposition); logm = 5 at c = 17 forces the tree
    for c, S, G, logm in ((2, 9, 4, 1), (3, 5, 4, 2), (4, 5, 4, 1), (7, 16, 4, 2), (8, 64, 16, 3), (11, 33, 16, 3),
                          (13, 7, 5, 3), (16, 50, 16, 2), (17, 64, 16, 3), (18, 64, 16, 2), (17, 64, 16, 14)):
        if c >= 15 and not table:
            continue  # W bucket sets of 2^14+ buckets: too slow for the CPU loop; the table layout covers the path
        assert _msm(emul, cid, table, c, S, G, logm, pts, sc) == want, (c, S, G, logm)
    assert _msm(emul, cid, table, 8, 16, 4, 3, pts, sc, is_mont=0) == want


def test_msm_case_families_hit_their_branches():
    """Each scalar family of tests/msm_cases.py reaches the recoding branch it is named for, at every window size."""
    for c in range(2, 25):
        K, B = 254 // c, 1 << (c - 1)
        for order in (O.PALLAS.order, O.VESTA.order):
            fam = families(c, order)
            dg, cin = signed_digits(fam["top_bucket"], c)
            assert dg[:K] == [B] * K and not any(cin)
            dg, cin = signed_digits(fam["neg_chain"], c)
            assert all(x <= 0 for x in dg[:K]) and all(cin[1:K + 1])
            dg, cin = signed_digits(fam["zero_with_carry"], c)
            assert dg[0] == -1 and dg[1:K] == [0] * (K - 1) and all(cin[1:K + 1]) and dg[K] == 1
            assert any(x == 0 and ci for x, ci in zip(*signed_digits(fam["zero_with_carry_254"], c)))
            for d in {1, B - 1, B}:
                dg, cin = signed_digits(fam[f"one_digit_{d}"], c)
                assert dg[:K] == [d] * K and not any(dg[K:]) and not any(cin)
            for d in {1, B - 1}:
                dg, cin = signed_digits(fam[f"alt_sign_{d}"], c)
                assert dg[:K - 1] == [-d] * (K - 1) and dg[K - 1] == d and not any(dg[K:])
            for name in ("order-1", "order-2", "half", "2^253", "2^254-B", "zero", "one"):
                signed_digits(fam[name], c)


def test_msm_digit_families(emul):
    """The scalar families through the emulated pipeline at every window size: c = 2..24 in the table layout (one
    bucket set), c = 2..10 in the plain layout (W sets), Montgomery and raw scalars, logm 3 and 8 (stage 6 takes the
    tree, the latency or the hybrid path), without and with batched-affine halving rounds."""
    k0, d = 3, 7
    pts = {cid: O.CURVES[cid].progression(k0, d, 24) for cid in (O.CURVE_PALLAS, O.CURVE_VESTA)}
    settings = ((1, 3, (0, 0)), (0, 8, (2, 5)))   # (is_mont, logm, affine rounds and K)
    try:
        for table, cs in ((1, range(2, 25)), (0, range(2, 11))):
            for c in cs:
                for cid in (O.CURVE_PALLAS, O.CURVE_VESTA):
                    cv = O.CURVES[cid]
                    sc = list(families(c, cv.order).values())
                    sc += rand_scalars(O.XorShiftRng(), cv.order, 24 - len(sc))
                    is_mont, logm, aff = settings[(c + cid) % 2]
                    emul.emul_set_affine(*aff)
                    got = _msm(emul, cid, table, c, 3, 4, logm, pts[cid], sc, is_mont)
                    assert got == O.jac_to_bytes(cv, cv.msm_known_dlog(sc, k0, d)), (table, c, cid, is_mont, logm)
    finally:
        emul.emul_set_affine(0, 0)


def test_msm_skewed_and_edges(emul):
    cv = O.PALLAS
    rng, py = O.XorShiftRng(), random.Random(1)
    n = 600
    pts = cv.progression(3, 5, n)
    sc = nova_like_scalars(py, rng, cv.order, n)
    want = O.jac_to_bytes(cv, cv.msm_known_dlog(sc, 3, 5))
    for table in (0, 1):
        for c, S, G in ((6, 4, 4), (9, 8, 5)):   # tiny S: > 4096 records -> record levels run
            assert _msm(emul, 0, table, c, S, G, 2, pts, sc) == want
    try:   # record levels in groups of 32 records (host mirror of the warp-cooperative level)
        for mode in (1, 2):    # 2: per-bucket record reduction (RecBucketFn, opt-in in the product)
            emul.emul_set_recwarp(mode)
            for table in (0, 1):
                for c, S in ((6, 4), (9, 2), (4, 3)):
                    assert _msm(emul, 0, table, c, S, 4, 2, pts, sc) == want
    finally:
        emul.emul_set_recwarp(0)
    assert _msm(emul, 0, 0, 8, 16, 4, 3, [], []) == bytes(96)
    assert _msm(emul, 0, 0, 8, 16, 4, 3, pts[:1], [0]) == bytes(96)
    assert _msm(emul, 0, 1, 8, 16, 4, 3, pts[:1], [5]) == O.jac_to_bytes(cv, cv.mul(5, pts[0]))
    # all scalars equal, all points equal: everything lands in the same buckets
    assert _msm(emul, 0, 0, 5, 8, 4, 2, [pts[4]] * 64, [12345] * 64) == O.jac_to_bytes(cv, cv.mul(12345 * 64, pts[4]))


def test_point_sum(emul):
    cv = O.VESTA
    pts = cv.progression(2, 9, 5) + [None]
    buf = aligned(b"".join(O.jac_to_bytes(cv, p) for p in pts))
    out = np.zeros(96, np.uint8)
    emul.emul_point_sum(1, ptr(buf), SZ(len(pts)), ptr(out))
    want = None
    for p in pts:
        want = cv.add(want, p)
    assert out.tobytes() == O.jac_to_bytes(cv, want)


@pytest.mark.parametrize("fid,mk", [(O.FIELD_FQ, O.PallasVDF), (O.FIELD_FP, O.VestaVDF)])
def test_minroot_check(emul, fid, mk):
    vdf = mk()
    rng = O.XorShiftRng()
    n = 64
    res, orig, ts = [], [], []
    for k in range(n):
        r = O.State(*rand_scalars(rng, vdf.m, 3))
        t = [0, 1, 2, 7, 10][k % 5]
        o = vdf.inverse_eval(r, t)
        if k % 9 == 4:
            o = O.State(o.x, o.y, (o.i + 1) % vdf.m)
        res.append(r); orig.append(o); ts.append(t)
    rb = aligned(b"".join(O.state_to_bytes(s, vdf.m) for s in res))
    ob = aligned(b"".join(O.state_to_bytes(s, vdf.m) for s in orig))
    tb = np.array(ts, dtype=np.uint64)
    ok = np.zeros(n, np.uint8)
    emul.emul_minroot_check(fid, ptr(rb), ptr(ob), ptr(tb), ctypes.c_uint64(0), SZ(n), ptr(ok))
    assert [bool(v) for v in ok] == [vdf.check(r, t, o) for r, t, o in zip(res, ts, orig)]
    out = np.zeros(n * 96, np.uint8)
    emul.emul_minroot_inverse_eval(fid, ptr(rb), ctypes.c_uint64(6), SZ(n), ptr(out))
    assert out.tobytes() == b"".join(O.state_to_bytes(vdf.inverse_eval(r, 6), vdf.m) for r in res)


@pytest.mark.parametrize("fid", [O.FIELD_FQ, O.FIELD_FP])
def test_r1cs_cross_term_and_fold(emul, fid):
    vdf = O.MinRootVDF(fid)
    m = vdf.m
    rng = O.XorShiftRng()
    t, aug = 6, 30
    s = vdf.eval(O.State(O.field_random(rng, m), 0, 1), t)
    shape, W1, X1, _ = O.make_step_instance(fid, t, s, aug_cons=aug)
    _, W2, X2, _ = O.make_step_instance(fid, t, vdf.eval(s, t), aug_cons=aug)
    coo = O.shape_to_coo_bytes(shape)
    keep = [aligned(x) for trip in coo for x in trip[:3]]
    args = []
    for k, trip in enumerate(coo):
        args += [ptr(keep[3 * k]), ptr(keep[3 * k + 1]), ptr(keep[3 * k + 2]), SZ(trip[3])]
    u1 = 0x1234567
    w1, w2 = aligned(O.fes_to_bytes(W1, m)), aligned(O.fes_to_bytes(W2, m))
    x1, x2, ub = aligned(O.fes_to_bytes(X1, m)), aligned(O.fes_to_bytes(X2, m)), aligned(O.fe_to_bytes(u1, m))
    out = np.zeros(3 * shape.num_cons * 32, np.uint8)
    assert emul.emul_r1cs(fid, 0, SZ(shape.num_cons), SZ(shape.num_vars), SZ(shape.num_io), *args,
                          ptr(w1), ptr(ub), ptr(x1), ptr(w2), ptr(x2), ptr(out)) == 0
    Az, Bz, Cz = shape.multiply_vec(shape.z_of(W1, u1, X1))
    assert O.fes_from_bytes(out.tobytes(), m) == Az + Bz + Cz
    assert emul.emul_r1cs(fid, 1, SZ(shape.num_cons), SZ(shape.num_vars), SZ(shape.num_io), *args,
                          ptr(w1), ptr(ub), ptr(x1), ptr(w2), ptr(x2), ptr(out)) == 0
    T = shape.cross_term(W1, u1, X1, W2, X2)
    assert O.fes_from_bytes(out.tobytes()[:shape.num_cons * 32], m) == T
    r = O.field_random(rng, m) >> 127
    E1 = rand_scalars(rng, m, shape.num_cons)
    e1, tb = aligned(O.fes_to_bytes(E1, m)), aligned(O.fes_to_bytes(T, m))
    emul.emul_fold(fid, ptr(w1), ptr(w2), SZ(len(W1)), ptr(e1), ptr(tb), SZ(len(E1)), ptr(aligned(O.fe_to_bytes(r, m))))
    assert O.fes_from_bytes(w1.tobytes(), m) == O.fold_vec(W1, W2, r, m)
    assert O.fes_from_bytes(e1.tobytes(), m) == O.fold_vec(E1, T, r, m)


@pytest.mark.parametrize("table", [0, 1])
def test_msm_batch(emul, table):
    """k scalar vectors of different lengths over the same generators in one pass (commit(W2), commit(T))."""
    cv = O.PALLAS
    rng, py = O.XorShiftRng(), random.Random(9)
    n = 150
    pts = cv.progression(8, 3, n)
    vecs = [rand_scalars(rng, cv.order, 150), nova_like_scalars(py, rng, cv.order, 97), [], [5]]
    for k in (1, 2, 4):
        use = vecs[:k]
        lens = np.array([len(v) for v in use], dtype=np.uint32)
        sb = aligned(b"".join(O.fes_to_bytes(v, cv.order) for v in use))
        out = np.zeros(96 * k, np.uint8)
        assert emul.emul_msm_batch(0, table, 7, 9, ptr(aligned(O.affines_to_bytes(cv, pts))), SZ(n), ptr(sb),
                                   ptr(lens), k, ptr(out)) == 0
        for j, v in enumerate(use):
            assert out.tobytes()[96 * j:96 * j + 96] == O.jac_to_bytes(cv, cv.msm_known_dlog(v, 8, 3)), (k, j)
    # the same batch with batched-affine halving rounds in front of the accumulation
    try:
        emul.emul_set_affine(2, 5)
        lens = np.array([len(v) for v in vecs], dtype=np.uint32)
        sb = aligned(b"".join(O.fes_to_bytes(v, cv.order) for v in vecs))
        out = np.zeros(96 * 4, np.uint8)
        assert emul.emul_msm_batch(0, table, 5, 9, ptr(aligned(O.affines_to_bytes(cv, pts))), SZ(n), ptr(sb),
                                   ptr(lens), 4, ptr(out)) == 0
        for j, v in enumerate(vecs):
            assert out.tobytes()[96 * j:96 * j + 96] == O.jac_to_bytes(cv, cv.msm_known_dlog(v, 8, 3)), j
    finally:
        emul.emul_set_affine(0, 0)


@pytest.mark.parametrize("table", [0, 1])
def test_msm_chunked(emul, table):
    """Point-range chunks accumulating into one bucket array (the host API's H2D/compute overlap schedule)."""
    cv = O.VESTA
    rng, py = O.XorShiftRng(), random.Random(21)
    n = 333
    pts = cv.progression(6, 13, n)
    pts[100] = None
    sc = nova_like_scalars(py, rng, cv.order, n)
    sc[5], sc[200] = cv.order - 1, 0
    want = O.jac_to_bytes(cv, cv.msm(sc, pts))
    for c, S, chunks in ((5, 7, 1), (5, 7, 2), (6, 16, 4), (9, 11, 8), (3, 5, 3)):
        out = np.zeros(96, np.uint8)
        assert emul.emul_msm_chunked(1, table, c, S, ptr(aligned(O.affines_to_bytes(cv, pts))), SZ(n),
                                     ptr(aligned(O.fes_to_bytes(sc, cv.order))), chunks, ptr(out)) == 0
        assert out.tobytes() == want, (c, S, chunks)
    try:   # chunks + affine rounds
        emul.emul_set_affine(3, 4)
        out = np.zeros(96, np.uint8)
        assert emul.emul_msm_chunked(1, table, 5, 7, ptr(aligned(O.affines_to_bytes(cv, pts))), SZ(n),
                                     ptr(aligned(O.fes_to_bytes(sc, cv.order))), 3, ptr(out)) == 0
        assert out.tobytes() == want
    finally:
        emul.emul_set_affine(0, 0)


@pytest.mark.parametrize("fid", [O.FIELD_FQ, O.FIELD_FP])
def test_minroot_step_witness(emul, fid):
    """Device witness generator vs the oracle's restatement of InverseMinRootCircuit::synthesize."""
    vdf = O.MinRootVDF(fid)
    rng = O.XorShiftRng()
    t, n = 9, 5
    res = [vdf.eval(O.State(O.field_random(rng, vdf.m), 0, 1), t) for _ in range(n)]
    out = np.zeros(n * (4 * t + 1) * 32, np.uint8)
    emul.emul_minroot_witness(fid, ptr(aligned(b"".join(O.state_to_bytes(s, vdf.m) for s in res))),
                              ctypes.c_uint64(t), SZ(n), ptr(out))
    got = O.fes_from_bytes(out.tobytes(), vdf.m)
    for k, s in enumerate(res):
        _, W, _, _ = O.make_step_instance(fid, t, s)
        assert got[k * (4 * t + 1):(k + 1) * (4 * t + 1)] == W[3:]   # W = [x, y, i | step variables]


@pytest.mark.parametrize("table", [0, 1])
def test_msm_affine_rounds(emul, table):
    """Batched-affine halving rounds (msm_affine.cuh) in front of the XYZZ accumulation: same result for any
    number of rounds, including the exceptional pairs (equal points -> doubling, P + (-P), identity operands)."""
    cv = O.PALLAS
    rng, py = O.XorShiftRng(), random.Random(7)
    n = 300
    pts = cv.progression(5, 11, n)
    sc = rand_scalars(rng, cv.order, n)
    sc[0], sc[1], sc[2] = 0, 1, cv.order - 1
    pts[7] = None                                      # identity operand
    for k in range(20, 40):                             # a run of equal points with equal scalars: doublings,
        pts[k], sc[k] = pts[20], sc[20]                 # then sums that meet again in later rounds
    for k in range(40, 50, 2):                          # P + (-P) in the same bucket
        pts[k + 1], sc[k + 1] = cv.neg(pts[k]), sc[k]
    want = O.jac_to_bytes(cv, cv.msm(sc, pts))
    skew = nova_like_scalars(py, rng, cv.order, n)
    want_skew = O.jac_to_bytes(cv, cv.msm(skew, pts))
    try:
        for rounds, K in ((1, 8), (2, 3), (3, 64), (6, 5), (2, 1)):
            emul.emul_set_affine(rounds, K)
            for c, S in ((4, 5), (7, 16), (11, 33)):
                assert _msm(emul, 0, table, c, S, 4, 2, pts, sc) == want, (rounds, K, c, S)
            assert _msm(emul, 0, table, 6, 4, 4, 2, pts, skew) == want_skew, (rounds, K)
        emul.emul_set_affine(2, 4)
        assert _msm(emul, 0, table, 5, 8, 4, 2, [pts[4]] * 64, [12345] * 64) == O.jac_to_bytes(cv, cv.mul(12345 * 64, pts[4]))
        assert _msm(emul, 0, table, 8, 16, 4, 3, pts[:1], [5]) == O.jac_to_bytes(cv, cv.mul(5, pts[0]))
        assert _msm(emul, 0, table, 8, 16, 4, 3, pts[:1], [0]) == bytes(96)
    finally:
        emul.emul_set_affine(0, 0)


@pytest.mark.parametrize("fid", [O.FIELD_FQ, O.FIELD_FP])
def test_r1cs_bind_rows(emul, fid):
    """ScaleRowsFn + BindRowsFn + BindHeavyFn (the inner sum-check's table) on the CPU against the oracle; t = 80 gives
    the constant column more than 64 entries, i.e. the heavy-column kernel runs."""
    vdf = O.MinRootVDF(fid)
    m = vdf.m
    rng = O.XorShiftRng()
    shape, W, X, _ = O.make_step_instance(fid, 80, O.State(3, 4, 80), aug_cons=25)
    coo = O.shape_to_coo_bytes(shape)
    keep = [aligned(x) for trip in coo for x in trip[:3]]
    args = []
    for k, trip in enumerate(coo):
        args += [ptr(keep[3 * k]), ptr(keep[3 * k + 1]), ptr(keep[3 * k + 2]), SZ(trip[3])]
    eq = rand_scalars(rng, m, shape.num_cons)
    r_abc = rand_scalars(rng, m, 3)
    eqb, rb = aligned(O.fes_to_bytes(eq, m)), aligned(O.fes_to_bytes(r_abc, m))
    dummy = aligned(bytes(32 * max(1, shape.num_io)))
    out = np.zeros((shape.num_vars + 1 + shape.num_io) * 32, np.uint8)
    heavy = emul.emul_r1cs(fid, 2, SZ(shape.num_cons), SZ(shape.num_vars), SZ(shape.num_io), *args,
                           ptr(eqb), ptr(rb), ptr(dummy), ptr(eqb), ptr(dummy), ptr(out))
    assert heavy >= 1
    assert O.fes_from_bytes(out.tobytes(), m) == shape.bind_rows(eq, r_abc)
