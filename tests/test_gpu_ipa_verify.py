"""GPU: batch verification of inner-product arguments (vdfgpu_ipa_verify_batch) on proofs from vdfgpu_ipa_prove:
verdicts against the reference at small sizes with random generators, one corrupted field at a time; corruptions that
cancel under equal weights; malformed and un-normalised points; known discrete logs at Nova sizes on both sides of the
MSM's graph-replay bound; the set layouts; two threads on their own streams; and the proof of the inner sum-check ->
IPA chain on a step instance."""
import hashlib
import random
import threading

import pytest

from oracle import pasta as O
from tests import ipa_ref as IR
from tests import ipa_verify_ref as VR
from tests import shape_gen as S
from vdf_b200 import _lib
from vdf_b200 import msm as G
from vdf_b200 import spartan as SP

pytestmark = pytest.mark.gpu

CIDS = [O.CURVE_PALLAS, O.CURVE_VESTA]
K0, D = 1234567, 89


def transcript(salt: bytes = b""):
    def ch(rnd, L, R):
        return int.from_bytes(hashlib.sha256(salt + bytes([rnd]) + L + R).digest(), "little")
    return ch


def random_set(cid, n, seed, **kw):
    cv = O.CURVES[cid]
    py = random.Random(seed)
    pts = [cv.mul(py.randrange(1, cv.order), cv.gen) for _ in range(n)]
    return pts, G.Generators.from_points(cid, pts, **kw)


def prove(g, cv, a, b, u_scale, salt, commit):
    """A proof tuple as spartan.ipa_verify_batch takes it; commit(a) gives comm_a as an affine point"""
    m = cv.order
    Ls, Rs, rs, a_hat = SP.ipa_prove(g, a, b, u_scale, transcript(salt))
    return (Ls, Rs, rs, a_hat, O.jac_to_bytes(cv, commit(a)), IR.inner(a, b, m), IR.inner(b, IR.s_table(rs, m), m),
            u_scale)


def to_ref(cv, p):
    """the proof with affine points, for tests/ipa_verify_ref.py"""
    Ls, Rs, rs, a_hat, comm, c, b_hat, u_scale = p
    pt = lambda x: O.jac_from_bytes(cv, x)  # noqa: E731
    return ([pt(x) for x in Ls], [pt(x) for x in Rs], rs, a_hat, pt(comm), c, b_hat, u_scale)


def corruptions(cv, p):
    """(name, proof) with one field of p changed"""
    m = cv.order
    Ls, Rs, rs, a_hat, comm, c, b_hat, u_scale = p
    gen = cv.gen
    shift = lambda x: O.jac_to_bytes(cv, cv.add(O.jac_from_bytes(cv, x), gen))  # noqa: E731
    out = [("a_hat", (Ls, Rs, rs, (a_hat + 1) % m, comm, c, b_hat, u_scale)),
           ("comm_a", (Ls, Rs, rs, a_hat, shift(comm), c, b_hat, u_scale)),
           ("c", (Ls, Rs, rs, a_hat, comm, (c + 1) % m, b_hat, u_scale)),
           ("b_hat", (Ls, Rs, rs, a_hat, comm, c, (b_hat + 1) % m, u_scale)),
           ("u_scale", (Ls, Rs, rs, a_hat, comm, c, b_hat, (u_scale + 1) % m))]
    if Ls:
        j = len(Ls) - 1
        out += [("L_j", ([shift(Ls[0])] + list(Ls[1:]), Rs, rs, a_hat, comm, c, b_hat, u_scale)),
                ("L_j <-> R_j", (list(Ls[:j]) + [Rs[j]], list(Rs[:j]) + [Ls[j]], rs, a_hat, comm, c, b_hat, u_scale)),
                ("r_j", (Ls, Rs, [rs[0] % (m - 1) + 1] + list(rs[1:]), a_hat, comm, c, b_hat, u_scale))]
    return out


# ---- random sets: honest proofs, then one corrupted field of one proof -------------------------------------------
@pytest.mark.parametrize("cid", CIDS)
@pytest.mark.parametrize("ell", [0, 1, 2, 6])
@pytest.mark.parametrize("k", [1, 5])
def test_random_sets_one_corruption_at_a_time(gpu_lib, cid, ell, k):
    cv = O.CURVES[cid]
    m = cv.order
    n = 1 << ell
    py = random.Random(100 * ell + 10 * k + cid)
    pts, g = random_set(cid, n + 1, 7 + ell + cid)
    proofs, bs = [], []
    for q in range(k):
        a = [py.randrange(m) for _ in range(n)]
        b = [py.randrange(m) for _ in range(n)]
        proofs.append(prove(g, cv, a, b, py.randrange(1, m), bytes([q, ell]), lambda a: cv.msm_naive(a, pts[:n])))
        bs.append(b)
    for p, b in zip(proofs, bs):   # the honest proofs pass ipa_ref.verify (P = comm_a + c U)
        Ls, Rs, rs, a_hat, comm, c, _, u_scale = to_ref(cv, p)
        U = cv.mul(u_scale, pts[n])
        assert IR.verify(cv, pts[:n], pts[n], u_scale, cv.add(comm, cv.mul(c, U)), b, Ls, Rs, rs, a_hat)
    assert SP.ipa_verify_batch(g, proofs) == [True] * k
    bad = min(1, k - 1)
    for name, x in corruptions(cv, proofs[bad]):
        # at ell = 0, a_hat b_hat = c for an honest proof, so u_scale has no term left to corrupt: the reference decides
        want = VR.verify_one(cv, pts[:n], pts[n], to_ref(cv, x)) if ell <= 2 else False
        got = SP.ipa_verify_batch(g, proofs[:bad] + [x] + proofs[bad + 1:])
        assert got == [q != bad or want for q in range(k)], name
    g.close()


# ---- corruptions that cancel: why the weights are random -------------------------------------------------------
@pytest.mark.parametrize("cid", CIDS)
def test_cancelling_corruptions(gpu_lib, cid):
    """Proof 0 gets comm_a + D and proof 1 comm_a - D.  With w = (1, 1) the two errors cancel in the weighted sum and
    the batch passes: exactly the forgery random weights rule out.  With weights from `secrets` both are flagged."""
    cv = O.CURVES[cid]
    m = cv.order
    ell = 3
    n = 1 << ell
    py = random.Random(20 + cid)
    g = G.Generators.progression(cid, K0, D, n + 1, table=True)
    commit = lambda a: cv.mul(sum(x * (K0 + i * D) for i, x in enumerate(a)) % m, cv.gen)  # noqa: E731
    proofs = [prove(g, cv, [py.randrange(m) for _ in range(n)], [py.randrange(m) for _ in range(n)], 3, bytes([q]),
                    commit) for q in range(2)]
    delta = cv.mul(py.randrange(1, m), cv.gen)
    moved = []
    for p, dd in zip(proofs, (delta, cv.neg(delta))):
        moved.append(p[:4] + (O.jac_to_bytes(cv, cv.add(O.jac_from_bytes(cv, p[4]), dd)),) + p[5:])
    assert SP.ipa_verify_batch(g, moved, weights=[1, 1]) == [True, True]
    assert SP.ipa_verify_batch(g, moved) == [False, False]
    assert SP.ipa_verify_batch(g, proofs) == [True, True]
    g.close()


# ---- malformed and unusual points ------------------------------------------------------------------------------
def raw_verify(lib, g, ell, comm, Ls, Rs, rs, a_hat, c, b_hat, u_scale, w):
    """vdfgpu_ipa_verify_batch on byte strings: every argument already encoded, proof-major"""
    k = len(comm) // 96
    ok = bytearray(k)
    p = _lib.as_ptr
    _lib.check(lib.vdfgpu_ipa_verify_batch(g._h, ell, k, p(comm), p(Ls or bytes(96)), p(Rs or bytes(96)),
                                           p(rs or bytes(32)), p(a_hat), p(c), p(b_hat), p(u_scale), p(w), p(ok)))
    return list(ok)


def encode(cv, proofs, w):
    m = cv.order
    col = lambda i: O.fes_to_bytes([p[i] for p in proofs], m)  # noqa: E731
    return (b"".join(p[4] for p in proofs), b"".join(x for p in proofs for x in p[0]),
            b"".join(x for p in proofs for x in p[1]), O.fes_to_bytes([r for p in proofs for r in p[2]], m), col(3),
            col(5), col(6), col(7), O.fes_to_bytes(w, m))


@pytest.mark.parametrize("cid", CIDS)
def test_malformed_and_unnormalised_points(gpu_lib, cid):
    cv = O.CURVES[cid]
    m, p_ = cv.order, cv.base
    ell = 3
    n = 1 << ell
    py = random.Random(30 + cid)
    g = G.Generators.progression(cid, K0, D, n + 1, table=True)
    commit = lambda a: cv.mul(sum(x * (K0 + i * D) for i, x in enumerate(a)) % m, cv.gen)  # noqa: E731
    rnd = lambda: [py.randrange(m) for _ in range(n)]  # noqa: E731
    proofs = [prove(g, cv, rnd(), rnd(), py.randrange(1, m), bytes([q]), commit) for q in range(5)]
    # a = 0: comm_a and every L and R are the identity, c = a_hat = 0
    proofs.append(prove(g, cv, [0] * n, rnd(), 5, b"zero", commit))
    assert proofs[-1][4] == bytes(96) and set(proofs[-1][0]) == {bytes(96)}
    # a_L = 0: L_0 is the identity
    proofs.append(prove(g, cv, [0] * (n // 2) + rnd()[n // 2:], rnd(), 5, b"half", commit))
    assert proofs[-1][0][0] == bytes(96) and proofs[-1][1][0] != bytes(96)
    w = [py.randrange(1, m) for _ in proofs]
    comm, Ls, Rs, rs, a_hat, c, b_hat, u_scale, wb = encode(cv, proofs, w)
    comm, Ls, a_hat = bytearray(comm), bytearray(Ls), bytearray(a_hat)
    # proof 0: L_1 off the curve (y + 1)
    x, y = O.jac_from_bytes(cv, bytes(Ls[96:192]))
    Ls[96 + 32:96 + 64] = O.fe_to_bytes(y + 1, p_)
    # proof 1: comm_a with X = p (a coordinate >= p; the same value as 0 mod p)
    comm[96:128] = p_.to_bytes(32, "little")
    # proof 2: a_hat = the group order (non-canonical)
    a_hat[64:96] = m.to_bytes(32, "little")
    # proof 3: comm_a as an un-normalised Jacobian point (X z^2, Y z^3, z): accepted like its normalised form
    x, y = O.jac_from_bytes(cv, bytes(comm[288:384]))
    z = py.randrange(2, p_)
    comm[288:384] = O.fe_to_bytes(x * z * z, p_) + O.fe_to_bytes(y * z ** 3, p_) + O.fe_to_bytes(z, p_)
    # proof 4: comm_a's Z = p + 1 (non-canonical)
    comm[384 + 64:480] = (p_ + 1).to_bytes(32, "little")
    got = raw_verify(gpu_lib, g, ell, bytes(comm), bytes(Ls), Rs, rs, bytes(a_hat), c, b_hat, u_scale, wb)
    assert got == [0, 0, 0, 1, 0, 1, 1]
    # the same proofs well-formed all pass, and an all-malformed batch is all zero
    assert SP.ipa_verify_batch(g, proofs) == [True] * len(proofs)
    assert raw_verify(gpu_lib, g, ell, bytes(comm[:288]), bytes(Ls[:3 * 96 * ell]), Rs[:3 * 96 * ell],
                      rs[:3 * 32 * ell], bytes(a_hat[:96]), c[:96], b_hat[:96], u_scale[:96], wb[:96]) == [0, 0, 0]
    g.close()


# ---- known discrete logs at Nova sizes ---------------------------------------------------------------------------
@pytest.mark.parametrize("cid", CIDS)
@pytest.mark.parametrize("ell,k", [(13, 8), (17, 8), (20, 4)], ids=["ell13-graph", "ell17-direct", "ell20"])
def test_known_discrete_logs(gpu_lib, cid, ell, k):
    """Progression set G_i = (K0 + i D) G: comm_a from the discrete log of <a, G>, b an eq table with b_hat in closed
    form.  All accepted; one corrupted a_hat among them is the only rejection (the batch fails, the single-proof
    checks find it)."""
    cv = O.CURVES[cid]
    m = cv.order
    fid = O.FIELD_FQ if cid == O.CURVE_PALLAS else O.FIELD_FP
    n = 1 << ell
    py = random.Random(40 + ell + cid)
    g = G.Generators.progression(cid, K0, D, n + 1, table=True)
    logs = [(K0 + i * D) % m for i in range(n)]
    a = [py.randrange(m) for _ in range(n)]
    comm = O.jac_to_bytes(cv, cv.mul(IR.inner(a, logs, m), cv.gen))
    proofs = []
    for q in range(k):
        x = [py.randrange(m) for _ in range(ell)]
        b = SP.eq_evals(fid, x)
        u_scale = py.randrange(1, m)
        Ls, Rs, rs, a_hat = SP.ipa_prove(g, a, b, u_scale, transcript(bytes([q, ell])))
        proofs.append((Ls, Rs, rs, a_hat, comm, IR.inner(a, b, m), SP.ipa_b_hat(fid, rs, [(1, x)]), u_scale))
    assert SP.ipa_verify_batch(g, proofs) == [True] * k
    bad = k // 2
    p = proofs[bad]
    proofs[bad] = p[:3] + ((p[3] + 1) % m,) + p[4:]
    assert SP.ipa_verify_batch(g, proofs) == [q != bad for q in range(k)]
    g.close()


# ---- set layouts ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cid", CIDS)
def test_set_layouts_give_the_same_verdicts(gpu_lib, cid):
    cv = O.CURVES[cid]
    m = cv.order
    ell = 9
    n = 1 << ell
    py = random.Random(50 + cid)
    commit = lambda a: cv.mul(sum(x * (K0 + i * D) for i, x in enumerate(a)) % m, cv.gen)  # noqa: E731
    g0 = G.Generators.progression(cid, K0, D, n + 1, table=True)
    proofs = [prove(g0, cv, [py.randrange(m) for _ in range(n)], [py.randrange(m) for _ in range(n)], 11, bytes([q]),
                    commit) for q in range(3)]
    g0.close()
    p = proofs[2]
    proofs.append(p[:4] + (proofs[0][4],) + p[5:])   # another proof's commitment
    w = [py.randrange(1, m) for _ in proofs]
    for kw in ({"table": True}, {}, {"raw_jacobian": True}, {"table": True, "raw_jacobian": True}):
        g = G.Generators.progression(cid, K0, D, n + 1, **kw)
        assert SP.ipa_verify_batch(g, proofs, w) == [True, True, True, False], kw
        assert SP.ipa_verify_batch(g, proofs[:3], w[:3]) == [True] * 3, kw
        g.close()


# ---- two threads, each on its own stream -------------------------------------------------------------------------
def test_two_threads_on_their_own_streams(gpu_lib):
    import torch
    cid = O.CURVE_PALLAS
    cv = O.CURVES[cid]
    m = cv.order
    ell = 10
    n = 1 << ell
    py = random.Random(60)
    g = G.Generators.progression(cid, K0, D, n + 1, table=True)
    commit = lambda a: cv.mul(sum(x * (K0 + i * D) for i, x in enumerate(a)) % m, cv.gen)  # noqa: E731
    proofs = [prove(g, cv, [py.randrange(m) for _ in range(n)], [py.randrange(m) for _ in range(n)], 2, bytes([q]),
                    commit) for q in range(6)]
    batches = [proofs[:3], proofs[3:]]
    p = batches[1][1]
    batches[1][1] = p[:5] + ((p[5] + 1) % m,) + p[6:]
    want = [[True] * 3, [True, False, True]]
    got = [None, None]
    errors = []
    start = threading.Barrier(2)

    def run(t):
        try:
            s = torch.cuda.Stream()
            _lib.check(gpu_lib.vdfgpu_set_stream(s.cuda_stream))
            start.wait()
            for _ in range(3):
                v = SP.ipa_verify_batch(g, batches[t])
                assert got[t] is None or v == got[t]
                got[t] = v
        except Exception as e:   # surfaces in the main thread
            errors.append(e)
        finally:
            _lib.check(gpu_lib.vdfgpu_set_stream(None))

    threads = [threading.Thread(target=run, args=(t,)) for t in range(2)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors
    assert got == want
    g.close()


# ---- end to end: the IPA proof of the inner sum-check -> IPA chain on a step instance ----------------------------
def transcript_sc(m):
    def ch(rnd, evals):
        return (sum(evals) * 0x9E3779B97F4A7C15 + rnd + 4242) % m
    return ch


def test_step_instance_proof_is_accepted(gpu_lib):
    """The flow of test_gpu_ipa.py::test_inner_sumcheck_then_ipa_on_a_step_instance (W padded to 2^12, the inner
    sum-check gives r_y, the IPA proves W(r_y[1:]) = <W, eq(r_y[1:])>), then verified here with b_hat in closed form
    from r_y[1:]; a copy with a tampered claim is rejected."""
    from vdf_b200 import nova as N
    cid, fid = O.CURVE_PALLAS, O.FIELD_FQ
    cv, m = O.CURVES[cid], O.Q
    ell = 12
    n = 1 << ell
    py = random.Random(900)
    shape, W, X = S.io_bound_step(fid, 600, O.State(3, 4, 600), 0)
    assert n // 2 < shape.num_vars <= n and shape.is_sat_relaxed(W, [0] * shape.num_cons, 1, X)
    gs = N.R1CSShape(fid, shape.num_cons, shape.num_vars, shape.num_io, shape.A, shape.B, shape.C)
    ell_x = (shape.num_cons - 1).bit_length()
    rx = [py.randrange(m) for _ in range(ell_x)]
    r_abc = [py.randrange(m) for _ in range(3)]
    Mt = gs.bind_rows(SP.eq_evals(fid, rx)[:shape.num_cons], r_abc)
    v = shape.num_vars
    pad = lambda t, k: list(t) + [0] * (k - len(t))  # noqa: E731
    Wp = pad(W, n)
    z = Wp + pad([1] + list(X), n)
    Mz = pad(Mt[:v], n) + pad(Mt[v:], n)
    _, ry, _ = SP.sumcheck(fid, [Mz, z], transcript_sc(m))
    w_eval = O.poly_evaluate(Wp, ry[1:], m)
    g = G.Generators.progression(cid, K0, D, n + 1, table=True)
    u_scale = py.randrange(1, m)
    Ls, Rs, rs, a_hat = SP.ipa_prove(g, Wp, SP.eq_evals(fid, ry[1:]), u_scale, transcript(b"nova"))
    comm = O.jac_to_bytes(cv, g.commit(Wp + [0]))
    proof = (Ls, Rs, rs, a_hat, comm, w_eval, SP.ipa_b_hat(fid, rs, [(1, ry[1:])]), u_scale)
    assert SP.ipa_verify_batch(g, [proof]) == [True]
    tampered = proof[:5] + ((w_eval + 1) % m,) + proof[6:]
    assert SP.ipa_verify_batch(g, [tampered]) == [False]
    assert SP.ipa_verify_batch(g, [tampered, proof]) == [False, True]
    gs.close()
    g.close()
