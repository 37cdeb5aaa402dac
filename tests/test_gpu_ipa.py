"""GPU: the whole inner-product argument on a resident generator set (vdfgpu_ipa_prove[_dev], vdfgpu_ipa_gens_hat)
against tests/ipa_ref.py: every L_j and R_j the callback sees and a_hat, byte for byte at small sizes with random
generators, by known discrete logs at Nova sizes on both sides of the MSM's graph-replay bound; the set layouts; the
host and device forms, the latter on a delayed caller stream; edge cases; and the chain inner sum-check -> IPA on a step
instance."""
import hashlib
import random

import pytest

from oracle import pasta as O
from tests import ipa_ref as IR
from tests import shape_gen as S
from vdf_b200 import VdfGpuError, _lib
from vdf_b200 import msm as G
from vdf_b200 import spartan as SP

pytestmark = pytest.mark.gpu

CIDS = [O.CURVE_PALLAS, O.CURVE_VESTA]
K0, D = 1234567, 89
GRAPH_MAX_ENTRIES = 1 << 22   # vdf_b200/csrc/api_core.cu: sorted entries up to which an MSM is replayed as a graph


def transcript(salt: bytes = b""):
    """A deterministic stand-in for nova's transcript: r from the round and the two points."""
    def ch(rnd, L, R):
        return int.from_bytes(hashlib.sha256(salt + bytes([rnd]) + L + R).digest(), "little")
    return ch


def random_set(cid, n, seed, **kw):
    cv = O.CURVES[cid]
    py = random.Random(seed)
    pts = [cv.mul(py.randrange(1, cv.order), cv.gen) for _ in range(n)]
    return pts, G.Generators.from_points(cid, pts, **kw)


def point(cv, b):
    return O.jac_from_bytes(cv, b)


# ---- small sizes, byte for byte --------------------------------------------------------------------------------
@pytest.mark.parametrize("cid", CIDS)
@pytest.mark.parametrize("ell", [0, 1, 2, 6])
def test_small_sizes_match_reference(gpu_lib, cid, ell):
    cv = O.CURVES[cid]
    m = cv.order
    n = 1 << ell
    py = random.Random(100 + 10 * ell + cid)
    pts, g = random_set(cid, n + 1, 200 + ell + cid)
    a = [py.randrange(m) for _ in range(n)]
    b = [py.randrange(m) for _ in range(n)]
    u_scale = py.randrange(1, m)
    ch = transcript(bytes([ell, cid]))
    Ls, Rs, rs, a_hat = SP.ipa_prove(g, a, b, u_scale, ch)
    wL, wR, wrs, w_hat = IR.prove(cv, pts[:n], pts[n], u_scale, a, b, ch)
    assert Ls == [O.jac_to_bytes(cv, p) for p in wL]
    assert Rs == [O.jac_to_bytes(cv, p) for p in wR]
    assert rs == wrs and a_hat == w_hat
    if ell == 0:
        assert a_hat == a[0] and Ls == []
    U0 = pts[n]
    P = cv.add(cv.msm_naive(a, pts[:n]), cv.mul(IR.inner(a, b, m) * u_scale, U0))
    pL, pR = [point(cv, x) for x in Ls], [point(cv, x) for x in Rs]
    assert IR.verify(cv, pts[:n], U0, u_scale, P, b, pL, pR, rs, a_hat)
    assert not IR.verify(cv, pts[:n], U0, u_scale, P, b, pL, pR, rs, (a_hat + 1) % m)
    if ell:
        assert not IR.verify(cv, pts[:n], U0, u_scale, P, b, pR, pL, rs, a_hat)
    # the verifier's folded generator
    assert point(cv, SP.ipa_gens_hat(g, rs)) == cv.msm_naive(IR.s_table(rs, m), pts[:n])
    g.close()


# ---- known discrete logs at Nova sizes ---------------------------------------------------------------------------
def _msm_path(g, n):
    """which side of the graph-replay bound the round's batched MSM (2 vectors of n + 1 scalars) lands on: the library
    exposes no replay counter, so this restates msm_dispatch's condition (api_core.cu: plan entries n W batch against
    GRAPH_MAX_ENTRIES, W = ceil(256 / c)) from the window size the set reports"""
    windows = -(-256 // g.window_bits(n + 1))
    return "graph" if (n + 1) * windows * 2 <= GRAPH_MAX_ENTRIES else "direct"


def _check_dlog(cv, ell, u_scale, a, b, Ls, Rs, rs):
    tr = IR.DlogTracker(cv, K0, D, ell, u_scale, a, b)
    for j, r in enumerate(rs):
        logL, logR = tr.round(r)
        assert Ls[j] == O.jac_to_bytes(cv, tr.point(logL)), j
        assert Rs[j] == O.jac_to_bytes(cv, tr.point(logR)), j
    return tr


@pytest.mark.parametrize("cid", CIDS)
@pytest.mark.parametrize("ell,path", [(13, "graph"), (17, "direct")], ids=["ell13-graph", "ell17-direct"])
def test_known_discrete_logs(gpu_lib, cid, ell, path):
    cv = O.CURVES[cid]
    m = cv.order
    n = 1 << ell
    py = random.Random(300 + ell + cid)
    g = G.Generators.progression(cid, K0, D, n + 1, table=True)
    assert _msm_path(g, n) == path
    a = [py.randrange(m) for _ in range(n)]
    b = [py.randrange(m) for _ in range(n)]
    u_scale = py.randrange(1, m)
    Ls, Rs, rs, a_hat = SP.ipa_prove(g, a, b, u_scale, transcript(bytes([ell])))
    tr = _check_dlog(cv, ell, u_scale, a, b, Ls, Rs, rs)
    assert tr.a == [a_hat]
    if ell < 17:
        return
    s = IR.coef_tables(rs, m)[-1]
    logs = [(K0 + i * D) % m for i in range(n)]
    G_hat = point(cv, SP.ipa_gens_hat(g, rs))
    assert G_hat == tr.point(IR.inner(s, logs, m))
    # the full verifier equation, P = commit(a) computed by the library
    U = tr.point(tr.u)
    P = cv.add(g.commit(a + [0]), cv.mul(IR.inner(a, b, m), U))
    for L, R, r in zip(Ls, Rs, rs):
        ri = pow(r, -1, m)
        P = cv.add(cv.add(cv.mul(r * r, point(cv, L)), P), cv.mul(ri * ri, point(cv, R)))
    assert P == cv.mul(a_hat, cv.add(G_hat, cv.mul(IR.inner(b, s, m), U)))
    g.close()


# ---- set layouts ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cid", CIDS)
def test_plain_and_raw_jacobian_sets_give_the_table_bytes(gpu_lib, cid):
    cv = O.CURVES[cid]
    m = cv.order
    ell = 9
    n = 1 << ell
    py = random.Random(400 + cid)
    a = [py.randrange(m) for _ in range(n)]
    b = [py.randrange(m) for _ in range(n)]
    u_scale = py.randrange(1, m)
    outs = []
    for kw in ({"table": True}, {}, {"raw_jacobian": True}, {"table": True, "raw_jacobian": True}):
        g = G.Generators.progression(cid, K0, D, n + 1, **kw)
        got = SP.ipa_prove(g, a, b, u_scale, transcript())
        outs.append((got, SP.ipa_gens_hat(g, got[2])))
        g.close()
    assert all(o == outs[0] for o in outs)
    _check_dlog(cv, ell, u_scale, a, b, *outs[0][0][:3])


# ---- host and device forms -------------------------------------------------------------------------------------
def _dev(b):
    import torch
    return torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()


@pytest.mark.parametrize("cid", CIDS)
def test_host_and_device_forms_agree(gpu_lib, cid):
    import torch
    cv = O.CURVES[cid]
    m = cv.order
    ell = 11
    n = 1 << ell
    py = random.Random(500 + cid)
    g = G.Generators.progression(cid, K0, D, n + 1, table=True)
    a = [py.randrange(m) for _ in range(n)]
    b = [py.randrange(m) for _ in range(n)]
    host = SP.ipa_prove(g, a, b, 7, transcript())
    ta, tb = _dev(O.fes_to_bytes(a, m)), _dev(O.fes_to_bytes(b, m))
    torch.cuda.synchronize()
    dev = SP.ipa_prove_dev(g, ta, tb, 7, transcript())
    assert dev == host
    _check_dlog(cv, ell, 7, a, b, *host[:3])
    g.close()


@pytest.fixture
def caller_stream(gpu_lib):
    """A caller-owned stream set for this thread, reset to the library stream afterwards."""
    import torch
    s = torch.cuda.Stream()
    try:
        yield s
    finally:
        torch.cuda.synchronize()
        _lib.check(gpu_lib.vdfgpu_set_stream(None))


def _sleep_ms(s, ms):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(s):
        a.record()
        torch.cuda._sleep(1_000_000)
        b.record()
    b.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(1_000_000 * ms / max(a.elapsed_time(b), 1e-3)))


def test_dev_form_on_a_delayed_caller_stream(gpu_lib, caller_stream):
    """The inputs hold stale vectors until the caller stream, behind a ~25 ms device delay, copies the fresh ones in;
    nothing synchronises in between, so work enqueued on any other stream would read the stale vectors."""
    import torch
    cid = O.CURVE_PALLAS
    cv = O.CURVES[cid]
    m = cv.order
    ell = 10
    n = 1 << ell
    py = random.Random(600)
    g = G.Generators.progression(cid, K0, D, n + 1, table=True)
    stale = [[py.randrange(m) for _ in range(n)] for _ in range(2)]
    fresh = [[py.randrange(m) for _ in range(n)] for _ in range(2)]
    ins = [_dev(O.fes_to_bytes(v, m)) for v in stale]
    srcs = [_dev(O.fes_to_bytes(v, m)) for v in fresh]
    s = caller_stream
    _lib.check(gpu_lib.vdfgpu_set_stream(s.cuda_stream))
    SP.ipa_prove_dev(g, ins[0], ins[1], 3, transcript())      # warm-up: modules, workspaces (consumes the stale vectors)
    for t, v in zip(ins, stale):
        t.copy_(_dev(O.fes_to_bytes(v, m)))
    torch.cuda.synchronize()
    _sleep_ms(s, 25)
    with torch.cuda.stream(s):
        for dst, src in zip(ins, srcs):
            dst.copy_(src)
    got = SP.ipa_prove_dev(g, ins[0], ins[1], 3, transcript())
    assert got == SP.ipa_prove(g, fresh[0], fresh[1], 3, transcript())
    _check_dlog(cv, ell, 3, fresh[0], fresh[1], *got[:3])
    g.close()


# ---- edge cases ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cid", CIDS)
def test_edge_cases(gpu_lib, cid):
    cv = O.CURVES[cid]
    m = cv.order
    ell = 5
    n = 1 << ell
    py = random.Random(700 + cid)
    pts, g = random_set(cid, n + 1, 800 + cid)
    a = [py.randrange(m) for _ in range(n)]
    b = [py.randrange(m) for _ in range(n)]
    # a_L = 0, hence c_L = 0: L_0 is the identity
    a0 = [0] * (n // 2) + a[n // 2:]
    Ls, Rs, rs, a_hat = SP.ipa_prove(g, a0, b, 3, transcript())
    assert Ls[0] == bytes(96) and Rs[0] != bytes(96)
    assert (Ls, Rs, rs, a_hat) == _ref_bytes(cv, pts, n, 3, a0, b, transcript())
    # r = 1 and r = order - 1 in every round
    for r in (1, m - 1):
        got = SP.ipa_prove(g, a, b, 1, lambda rnd, L, R, r=r: r)
        assert got == _ref_bytes(cv, pts, n, 1, a, b, lambda rnd, L, R, r=r: r)
    # b = an eq table from the library, the real use
    fid = O.FIELD_FQ if cid == O.CURVE_PALLAS else O.FIELD_FP
    eq = SP.eq_evals(fid, [py.randrange(m) for _ in range(ell)])
    got = SP.ipa_prove(g, a, eq, 9, transcript())
    assert got == _ref_bytes(cv, pts, n, 9, a, eq, transcript())
    # a failing callback and one that returns 0: VDFGPU_ERR_STATE, and the next call works
    def boom(rnd, L, R):
        raise RuntimeError("transcript failed")
    for bad in (boom, lambda rnd, L, R: 0 if rnd == 2 else 5):
        with pytest.raises(VdfGpuError) as e:
            SP.ipa_prove(g, a, b, 1, bad)
        assert e.value.code == -3
        assert SP.ipa_prove(g, a, b, 9, transcript()) == _ref_bytes(cv, pts, n, 9, a, b, transcript())
    # too few points for ell: an argument error
    with pytest.raises(VdfGpuError) as e:
        SP.ipa_prove(g, a + a, b + b, 1, transcript())
    assert e.value.code == -1
    g.close()


def _raw_call(lib, g, a, b, m, ell, write_r):
    """vdfgpu_ipa_prove with a C-level callback: write_r(round) returns the 32 raw bytes it writes as r"""
    import ctypes

    def fn(_user, rnd, _L, _R, r_out):
        ctypes.memmove(r_out, write_r(int(rnd)), 32)
        return 0
    cb = _lib.IPA_ROUND_FN(fn)
    a_hat = bytearray(32)
    rc = lib.vdfgpu_ipa_prove(g._h, _lib.as_ptr(O.fes_to_bytes(a, m)), _lib.as_ptr(O.fes_to_bytes(b, m)), ell,
                              _lib.as_ptr(O.fe_to_bytes(1, m)), ctypes.cast(cb, ctypes.c_void_p), None, _lib.as_ptr(a_hat))
    return rc, lib.vdfgpu_last_error().decode()


@pytest.mark.parametrize("cid", CIDS)
def test_non_canonical_challenges_and_a_set_in_use(gpu_lib, cid):
    """r = order (0 in disguise) and r = order + 1 written by a C-level callback end the call with VDFGPU_ERR_STATE;
    vdfgpu_ipa_gens_hat refuses them as argument errors; the set cannot be destroyed while a call uses it."""
    cv = O.CURVES[cid]
    m = cv.order
    ell = 4
    n = 1 << ell
    py = random.Random(1000 + cid)
    pts, g = random_set(cid, n + 1, 1100 + cid)
    a = [py.randrange(m) for _ in range(n)]
    b = [py.randrange(m) for _ in range(n)]
    good = O.fe_to_bytes(5, m)
    for bad in (m.to_bytes(32, "little"), (m + 1).to_bytes(32, "little"), bytes(32)):
        rc, msg = _raw_call(gpu_lib, g, a, b, m, ell, lambda rnd, bad=bad: bad if rnd == 1 else good)
        assert rc == -3 and "challenge" in msg, msg
        rs = (good + bad + good)
        out = bytearray(96)
        assert gpu_lib.vdfgpu_ipa_gens_hat(g._h, _lib.as_ptr(rs), 3, _lib.as_ptr(out)) == -1
    # destroying the set from inside the callback (between rounds, outside the library's lock) is refused
    seen = []

    def destroy_then_answer(rnd):
        seen.append(gpu_lib.vdfgpu_gens_destroy(g._h))
        return good
    rc, msg = _raw_call(gpu_lib, g, a, b, m, ell, destroy_then_answer)
    assert rc == 0, msg
    assert seen == [-3] * ell
    # the call has returned: the set is released, still correct, and can be destroyed
    assert SP.ipa_prove(g, a, b, 9, transcript()) == _ref_bytes(cv, pts, n, 9, a, b, transcript())
    assert gpu_lib.vdfgpu_gens_destroy(g._h) == 0
    g._h = None


def _ref_bytes(cv, pts, n, u_scale, a, b, ch):
    Ls, Rs, rs, a_hat = IR.prove(cv, pts[:n], pts[n], u_scale, a, b, ch)
    return [O.jac_to_bytes(cv, p) for p in Ls], [O.jac_to_bytes(cv, p) for p in Rs], rs, a_hat


# ---- the pipeline as nova runs it: inner sum-check, then the IPA on W ------------------------------------------
def test_inner_sumcheck_then_ipa_on_a_step_instance(gpu_lib):
    """z = [W | u | X] with W padded to 2^12 (nova pads the witness to a power of two), the inner quadratic sum-check
    over (M(r_x, .), z) gives r_y; z(r_y) = (1 - r_y[0]) W(r_y[1:]) + r_y[0] (u | X)(r_y[1:]), and the IPA proves
    W(r_y[1:]) = <W, eq(r_y[1:])> on Pallas: a = W, b = eq(r_y[1:])."""
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
    evals, ry, fin = SP.sumcheck(fid, [Mz, z], transcript_sc(m))
    assert fin[0] == O.poly_evaluate(Mz, ry, m) and len(evals) == ell + 1
    w_eval = O.poly_evaluate(Wp, ry[1:], m)
    io_eval = O.poly_evaluate(pad([1] + list(X), n), ry[1:], m)
    assert fin[1] == ((1 - ry[0]) * w_eval + ry[0] * io_eval) % m
    b = SP.eq_evals(fid, ry[1:])
    assert IR.inner(Wp, b, m) == w_eval
    g = G.Generators.progression(cid, K0, D, n + 1, table=True)
    u_scale = py.randrange(1, m)
    Ls, Rs, rs, a_hat = SP.ipa_prove(g, Wp, b, u_scale, transcript(b"nova"))
    tr = _check_dlog(cv, ell, u_scale, Wp, b, Ls, Rs, rs)
    assert tr.a == [a_hat]
    s = IR.coef_tables(rs, m)[-1]
    U = tr.point(tr.u)
    P = cv.add(g.commit(Wp + [0]), cv.mul(w_eval, U))
    for L, R, r in zip(Ls, Rs, rs):
        ri = pow(r, -1, m)
        P = cv.add(cv.add(cv.mul(r * r, point(cv, L)), P), cv.mul(ri * ri, point(cv, R)))
    G_hat = point(cv, SP.ipa_gens_hat(g, rs))
    assert P == cv.mul(a_hat, cv.add(G_hat, cv.mul(IR.inner(b, s, m), U)))
    gs.close()
    g.close()


def transcript_sc(m):
    def ch(rnd, evals):
        return (sum(evals) * 0x9E3779B97F4A7C15 + rnd + 4242) % m
    return ch

