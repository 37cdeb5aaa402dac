"""GPU: the R1CS entry points on the general shapes of tests/shape_gen.py (constraints that read X, zero coefficients,
repeated pairs, empty and long rows, columns of exactly 64 and 65 entries, num_io 0, 2 and 7), on the IO-bound step
instance along a fold chain, and on a 2^18-constraint shape whose X columns are heavy -- host and device-pointer forms,
against the oracle."""
import random

import pytest

from oracle import pasta as O
from tests import shape_gen as S
from tests.sat_ref import unsat_rows
from vdf_b200 import _lib
from vdf_b200 import msm as G
from vdf_b200 import nova as N

pytestmark = pytest.mark.gpu

FIELD_CURVE = [(O.FIELD_FQ, O.CURVE_PALLAS), (O.FIELD_FP, O.CURVE_VESTA)]
DIMS = [(517, 300, 0), (1337, 900, 2), (2003, 1500, 7)]
K0, D = 3131, 19


def _gpu_shape(fid, shape):
    return N.R1CSShape(fid, shape.num_cons, shape.num_vars, shape.num_io, shape.A, shape.B, shape.C)


def _report(rep):
    return rep.bad_rows, rep.first_bad_row


def _want(shape, W, E, u, X):
    bad = unsat_rows(shape, W, E, u, X)
    return len(bad), (bad[0] if bad else None)


@pytest.mark.parametrize("fid,cid", FIELD_CURVE)
@pytest.mark.parametrize("cons,vars_,io", DIMS)
def test_host_entry_points(gpu_lib, fid, cid, cons, vars_, io):
    cv = O.CURVES[cid]
    shape = S.general_shape(fid, cons, vars_, io)
    m = shape.m
    gs = _gpu_shape(fid, shape)
    py = random.Random(cons * 3 + io)
    W1, X1, u1 = S.random_vec(py, m, vars_), S.random_vec(py, m, io), py.randrange(2, m)
    W2, X2 = S.random_vec(py, m, vars_), S.random_vec(py, m, io)
    z = shape.z_of(W1, u1, X1)
    assert list(gs.multiply_vec(z)) == shape.multiply_vec(z)
    gens = G.Generators.progression(cid, K0, D, max(cons, vars_), table=True)
    T, cT = gs.commit_T(gens, W1, u1, X1, W2, X2)
    assert T == shape.cross_term(W1, u1, X1, W2, X2)
    assert cT == cv.msm_known_dlog(T, K0, D)
    eq = S.random_vec(py, m, cons)
    for r_abc in ([py.randrange(m) for _ in range(3)], [0, 1, m - 1]):
        assert gs.bind_rows(eq, r_abc) == shape.bind_rows(eq, r_abc)
    # satisfiability: exact count and first row, commitments by the known-discrete-log identity
    W, E, u, X = S.relaxed_instance(shape)
    U = N.RelaxedR1CSInstance(cv.msm_known_dlog(W, K0, D), cv.msm_known_dlog(E, K0, D), list(X), u)
    rep = gs.is_sat_relaxed(gens, W, E, U)
    assert (rep.bad_rows, rep.first_bad_row, rep.comm_W_ok, rep.comm_E_ok) == (0, None, True, True)
    for j in range(io):   # one X entry only
        X2_ = list(X)
        X2_[j] = (X2_[j] + 1) % m
        rep = gs.is_sat_relaxed(gens, W, E, N.RelaxedR1CSInstance(U.comm_W, U.comm_E, X2_, u))
        assert _report(rep) == _want(shape, W, E, u, X2_) and rep.bad_rows > 0
        assert (rep.comm_W_ok, rep.comm_E_ok) == (True, True)
    E2 = list(E)
    E2[cons - 1] = (E2[cons - 1] + 1) % m
    rep = gs.is_sat_relaxed(None, W, E2, N.RelaxedR1CSInstance(None, None, list(X), u))
    assert _report(rep) == (1, cons - 1)
    # fold of W, E with r = 0, m - 1 and a 128-bit challenge
    for r in (0, m - 1, py.randrange(1 << 128)):
        assert N.fold_vectors(fid, W1, W2, E, T, r) == (O.fold_vec(W1, W2, r, m), O.fold_vec(E, T, r, m))
    gs.close()


def _dev(vals, m):
    import torch
    return torch.frombuffer(bytearray(O.fes_to_bytes(vals, m) or bytes(32)), dtype=torch.uint8).cuda()


def _host(t, m):
    return O.fes_from_bytes(t.cpu().numpy().tobytes(), m)


def _run(lib, fn, *args):
    """A _dev call on tensors written by torch: torch's stream is drained first, the library's stream after."""
    import torch
    torch.cuda.synchronize()
    _lib.check(fn(*args))
    _lib.check(lib.vdfgpu_synchronize())


@pytest.mark.parametrize("fid", [O.FIELD_FQ, O.FIELD_FP])
@pytest.mark.parametrize("cons,vars_,io", DIMS)
def test_dev_entry_points_equal_host_forms(gpu_lib, fid, cons, vars_, io):
    import torch
    lib = gpu_lib
    shape = S.general_shape(fid, cons, vars_, io)
    m = shape.m
    gs = _gpu_shape(fid, shape)
    h = gs._h
    py = random.Random(cons * 5 + io)
    W1, X1, u1 = S.random_vec(py, m, vars_), S.random_vec(py, m, io), py.randrange(2, m)
    W2, X2 = S.random_vec(py, m, vars_), S.random_vec(py, m, io)
    W1d, W2d, uX1d, uX2d = _dev(W1, m), _dev(W2, m), _dev([u1] + X1, m), _dev([1] + X2, m)
    ABC = torch.zeros(3 * cons * 32, dtype=torch.uint8, device="cuda")
    _run(lib, lib.vdfgpu_multiply_vec_dev, h, W1d.data_ptr(), uX1d.data_ptr(), ABC.data_ptr())
    Az, Bz, Cz = gs.multiply_vec(shape.z_of(W1, u1, X1))
    assert _host(ABC, m) == Az + Bz + Cz
    Td = torch.zeros(cons * 32, dtype=torch.uint8, device="cuda")
    _run(lib, lib.vdfgpu_cross_term_dev, h, W1d.data_ptr(), uX1d.data_ptr(), W2d.data_ptr(), uX2d.data_ptr(), Td.data_ptr())
    T, _ = gs.commit_T(None, W1, u1, X1, W2, X2)
    assert _host(Td, m) == T
    # bind_rows_dev: the scratch buffer holds the three scaled row tables (3 cons elements)
    eq, r_abc = S.random_vec(py, m, cons), [py.randrange(m) for _ in range(3)]
    scratch = torch.zeros(3 * cons * 32, dtype=torch.uint8, device="cuda")
    Mt = torch.zeros((vars_ + 1 + io) * 32, dtype=torch.uint8, device="cuda")
    eqd, rd = _dev(eq, m), _dev(r_abc, m)
    _run(lib, lib.vdfgpu_r1cs_bind_rows_dev, h, eqd.data_ptr(), rd.data_ptr(), scratch.data_ptr(), Mt.data_ptr())
    assert _host(Mt, m) == gs.bind_rows(eq, r_abc)
    # fold_dev over W and E in one launch; r on the device
    E1 = S.random_vec(py, m, cons)
    E1d = _dev(E1, m)
    r = py.randrange(1 << 128)
    _run(lib, lib.vdfgpu_fold_dev, fid, W1d.data_ptr(), W2d.data_ptr(), vars_, E1d.data_ptr(), Td.data_ptr(), cons,
         _dev([r], m).data_ptr())
    assert (_host(W1d, m), _host(E1d, m)) == N.fold_vectors(fid, W1, W2, E1, T, r)
    # is_sat_relaxed_dev: satisfied, and an X-only corruption
    W, E, u, X = S.relaxed_instance(shape)
    Wd, Ed = _dev(W, m), _dev(E, m)
    counts = torch.full((2,), -1, dtype=torch.int64, device="cuda")
    for X_ in ([X] + [[(x + 1) % m if k == j else x for k, x in enumerate(X)] for j in (0, io - 1)] if io else [X]):
        _run(lib, lib.vdfgpu_r1cs_is_sat_relaxed_dev, h, Wd.data_ptr(), Ed.data_ptr(), _dev([u] + X_, m).data_ptr(),
             counts.data_ptr())
        host = gs.is_sat_relaxed(None, W, E, N.RelaxedR1CSInstance(None, None, X_, u))
        assert counts.cpu().tolist() == [host.bad_rows, cons if host.first_bad_row is None else host.first_bad_row]
        assert _report(host) == _want(shape, W, E, u, X_)
    gs.close()


@pytest.mark.parametrize("fid,cid", FIELD_CURVE)
def test_running_chain_on_the_io_bound_shape(gpu_lib, fid, cid):
    """Three folds of fresh IO-bound instances (X2 different at every step): T (through comm_T and the folded E),
    both commitments, the folded W, E, u, X and the resident check after every step, and is_sat of every fresh one."""
    cv = O.CURVES[cid]
    t, aug = 5, 64
    shape, W0, X0 = S.fresh_instance(fid, t, 0, aug)
    m = shape.m
    gs = _gpu_shape(fid, shape)
    gens = G.Generators.progression(cid, K0, D, max(shape.num_cons, shape.num_vars), table=True)
    prover = N.RunningProver(gs, gens)
    prover.set_running(W0, [0] * shape.num_cons, N.RelaxedR1CSInstance(cv.msm_known_dlog(W0, K0, D), None, list(X0), 1))
    Wr, Er, ur, Xr = list(W0), [0] * shape.num_cons, 1, list(X0)
    seen = [X0]
    for k in range(1, 4):
        _, W2, X2 = S.fresh_instance(fid, t, k, aug)
        assert X2 not in seen
        seen.append(X2)
        rep = gs.is_sat(gens, W2, X2, cv.msm_known_dlog(W2, K0, D))
        assert (rep.bad_rows, rep.comm_W_ok) == (0, True)
        T_want = shape.cross_term(Wr, ur, Xr, W2, X2)
        assert T_want != shape.cross_term(Wr, ur, Xr, W2, Xr)   # T reads X2
        comm_T, r = prover.prove_step(W2, X2)
        assert comm_T == cv.msm_known_dlog(T_want, K0, D)
        Wr, Er = O.fold_vec(Wr, W2, r, m), O.fold_vec(Er, T_want, r, m)
        ur, Xr = (ur + r) % m, O.fold_vec(Xr, X2, r, m)
        assert prover.get_running() == (Wr, Er, ur, Xr)
        assert unsat_rows(shape, Wr, Er, ur, Xr) == []
        assert (prover.U.u, prover.U.X) == (ur, Xr)
        assert prover.U.comm_W == cv.msm_known_dlog(Wr, K0, D)
        assert prover.U.comm_E == cv.msm_known_dlog(Er, K0, D)
        rep = prover.check()
        assert (rep.bad_rows, rep.first_bad_row, rep.comm_W_ok, rep.comm_E_ok) == (0, None, True, True), k
    # a corrupted X1 in the fresh instance: exactly the IO-binding rows that read X1
    X_bad = [X0[0], (X0[1] + 1) % m]
    rep = gs.is_sat(None, W0, X_bad)
    assert _report(rep) == _want(shape, W0, None, 1, X_bad) == (3, shape.num_cons - 3)
    prover.close()


def test_fold_at_t1024_on_the_io_bound_shape(gpu_lib):
    """One fold of a fresh IO-bound instance into a relaxed running instance (u != 1, E != 0) at t = 1024 with the
    9800-constraint augmented block."""
    fid, cid = O.FIELD_FQ, O.CURVE_PALLAS
    cv = O.CURVES[cid]
    t, aug = 1024, 9800
    shape, W0, X0 = S.fresh_instance(fid, t, 0, aug)
    _, W1, X1 = S.fresh_instance(fid, t, 1, aug)
    _, W2, X2 = S.fresh_instance(fid, t, 2, aug)
    m = shape.m
    r0 = 0x1F2E3D4C5B6A79880123456789ABCDEF
    T0 = shape.cross_term(W0, 1, X0, W1, X1)
    Wr, Er = O.fold_vec(W0, W1, r0, m), O.fold_vec([0] * shape.num_cons, T0, r0, m)
    ur, Xr = (1 + r0) % m, O.fold_vec(X0, X1, r0, m)
    assert unsat_rows(shape, Wr, Er, ur, Xr) == [] and any(Er[-4:])
    gs = _gpu_shape(fid, shape)
    gens = G.Generators.progression(cid, K0, D, max(shape.num_cons, shape.num_vars), table=True)
    prover = N.RunningProver(gs, gens)
    prover.set_running(Wr, Er, N.RelaxedR1CSInstance(cv.msm_known_dlog(Wr, K0, D), cv.msm_known_dlog(Er, K0, D), Xr, ur))
    T_want = shape.cross_term(Wr, ur, Xr, W2, X2)
    comm_T, r = prover.prove_step(W2, X2)
    assert comm_T == cv.msm_known_dlog(T_want, K0, D)
    Wn, En = O.fold_vec(Wr, W2, r, m), O.fold_vec(Er, T_want, r, m)
    un, Xn = (ur + r) % m, O.fold_vec(Xr, X2, r, m)
    assert prover.get_running() == (Wn, En, un, Xn)
    rep = prover.check()
    assert (rep.bad_rows, rep.first_bad_row, rep.comm_W_ok, rep.comm_E_ok) == (0, None, True, True)
    prover.close()


def _hbm_like_shape(fid, log2rows):
    """bench.py's r1cs_hbm shape ("random_B": B holds a full-size coefficient) at 2^log2rows + 3 constraints, with X
    referenced: every fifth A row also reads an X column (two heavy columns of ~2^log2rows / 10 entries), B's columns
    run over W, u and X."""
    m = O.MODULUS[fid]
    cons, vars_, io = (1 << log2rows) + 3, 1 << log2rows, 2
    ncols = vars_ + 1 + io
    rnd = 0x1234567890ABCDEF1234567890ABCDEF
    A = [(r, r % vars_, 1) for r in range(cons)] + [(r, vars_ + 1 + (r // 5) % 2, m - 1) for r in range(0, cons, 5)]
    B = [(r, (r * 7 + 3) % ncols, rnd) for r in range(cons)]
    C = [(r, (r + 1) % vars_, 1) for r in range(cons)] + [(r, (r * 5) % vars_, m - 1) for r in range(cons)]
    return O.R1CSShape(m, cons, vars_, io, A, B, C)


def test_shape_at_2_18_constraints_with_x_columns(gpu_lib):
    import torch
    lib = gpu_lib
    fid = O.FIELD_FQ
    shape = _hbm_like_shape(fid, 18)
    m, cons, vars_, io = shape.m, shape.num_cons, shape.num_vars, shape.num_io
    gs = _gpu_shape(fid, shape)
    h = gs._h
    py = random.Random(18)
    W1, W2 = [py.randrange(m) for _ in range(vars_)], [py.randrange(m) for _ in range(vars_)]
    u1, X1, X2 = py.randrange(m), [py.randrange(m) for _ in range(io)], [py.randrange(m) for _ in range(io)]
    W1d, W2d, uX1d, uX2d = _dev(W1, m), _dev(W2, m), _dev([u1] + X1, m), _dev([1] + X2, m)
    ABC = torch.zeros(3 * cons * 32, dtype=torch.uint8, device="cuda")
    _run(lib, lib.vdfgpu_multiply_vec_dev, h, W1d.data_ptr(), uX1d.data_ptr(), ABC.data_ptr())
    Az, Bz, Cz = shape.multiply_vec(shape.z_of(W1, u1, X1))
    assert _host(ABC, m) == Az + Bz + Cz
    Td = torch.zeros(cons * 32, dtype=torch.uint8, device="cuda")
    _run(lib, lib.vdfgpu_cross_term_dev, h, W1d.data_ptr(), uX1d.data_ptr(), W2d.data_ptr(), uX2d.data_ptr(), Td.data_ptr())
    Az2, Bz2, Cz2 = shape.multiply_vec(shape.z_of(W2, 1, X2))
    assert _host(Td, m) == [(a1 * b2 + a2 * b1 - u1 * c2 - c1) % m
                            for a1, b1, c1, a2, b2, c2 in zip(Az, Bz, Cz, Az2, Bz2, Cz2)]
    eq, r_abc = [py.randrange(m) for _ in range(cons)], [py.randrange(m) for _ in range(3)]
    scratch = torch.zeros(3 * cons * 32, dtype=torch.uint8, device="cuda")
    Mt = torch.zeros((vars_ + 1 + io) * 32, dtype=torch.uint8, device="cuda")
    _run(lib, lib.vdfgpu_r1cs_bind_rows_dev, h, _dev(eq, m).data_ptr(), _dev(r_abc, m).data_ptr(), scratch.data_ptr(),
         Mt.data_ptr())
    assert _host(Mt, m) == shape.bind_rows(eq, r_abc)
    # relaxed instance of z1: E = Az.Bz - u1.Cz; then X1[1] corrupted
    E = [(a * b - u1 * c) % m for a, b, c in zip(Az, Bz, Cz)]
    counts = torch.full((2,), -1, dtype=torch.int64, device="cuda")
    Ed = _dev(E, m)
    for X_ in (X1, [X1[0], (X1[1] + 1) % m]):
        _run(lib, lib.vdfgpu_r1cs_is_sat_relaxed_dev, h, W1d.data_ptr(), Ed.data_ptr(), _dev([u1] + X_, m).data_ptr(),
             counts.data_ptr())
        bad = unsat_rows(shape, W1, E, u1, X_)
        assert counts.cpu().tolist() == [len(bad), bad[0] if bad else cons]
    assert counts.cpu().tolist()[0] > 10000
    gs.close()
