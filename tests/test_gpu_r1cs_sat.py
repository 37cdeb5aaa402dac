"""GPU: the satisfiability checks of RecursiveSNARK::verify (src/nova/proof.rs:382) -- is_sat_relaxed of the running
instances and is_sat of a fresh one -- through the C ABI, against the violating rows the oracle finds and the
known-discrete-log commitments: exact reports for corrupted instances, commitments compared as group elements,
the resident running instance checked in place along a fold chain, the device-pointer form, argument errors."""
import ctypes
import random
import subprocess

import pytest

from oracle import pasta as O
from tests.sat_ref import (build_sat_check, fresh_instance, hub_variable, relaxed_by_error, relaxed_instance,
                           sat_check_fixtures, unsat_rows)
from vdf_b200 import msm as G
from vdf_b200 import nova as N

pytestmark = pytest.mark.gpu

K0, D = 4242, 17


def _gpu_shape(fid, shape):
    return N.R1CSShape(fid, shape.num_cons, shape.num_vars, shape.num_io, shape.A, shape.B, shape.C)


def _want(shape, W, E, u, X):
    bad = unsat_rows(shape, W, E, u, X)
    return len(bad), (bad[0] if bad else None)


def _jac_unnormalised(cv, pt, z):
    """pt as a Jacobian point with Z = z != 1 (the same group element)."""
    m = cv.base
    return (O.fe_to_bytes(pt[0] * z * z, m) + O.fe_to_bytes(pt[1] * z * z * z, m) + O.fe_to_bytes(z, m))


@pytest.mark.parametrize("fid,cid", [(O.FIELD_FQ, O.CURVE_PALLAS), (O.FIELD_FP, O.CURVE_VESTA)])
def test_running_check_along_a_fold_chain(gpu_lib, fid, cid):
    """test_running_prover_chain's three folds (t = 5): after every step the resident instance and the downloaded
    vectors are both reported satisfied with both commitments equal."""
    cv = O.CURVES[cid]
    t, aug = 5, 64
    shape, W0, X0 = fresh_instance(fid, t, 0, aug)
    gs = _gpu_shape(fid, shape)
    gens = G.Generators.progression(cid, K0, D, max(shape.num_cons, shape.num_vars), table=True)
    prover = N.RunningProver(gs, gens)
    U = N.RelaxedR1CSInstance(comm_W=gens.commit(W0), comm_E=None, X=list(X0), u=1)
    prover.set_running(W0, [0] * shape.num_cons, U)
    rep = prover.check()
    assert (rep.bad_rows, rep.first_bad_row, rep.comm_W_ok, rep.comm_E_ok, rep.ok) == (0, None, True, None, True)
    for k in range(1, 4):
        _, W2, X2 = fresh_instance(fid, t, k, aug)
        prover.prove_step(W2, X2)
        rep = prover.check()
        assert (rep.bad_rows, rep.first_bad_row, rep.comm_W_ok, rep.comm_E_ok) == (0, None, True, True), k
        Wg, Eg, ug, Xg = prover.get_running()
        assert unsat_rows(shape, Wg, Eg, ug, Xg) == []
        assert prover.U.comm_E == cv.msm_known_dlog(Eg, K0, D)
        host = gs.is_sat_relaxed(gens, Wg, Eg, prover.U)
        assert host == rep and host.ok
    # a wrong commitment in the instance is caught in place
    prover.U = N.RelaxedR1CSInstance(comm_W=prover.U.comm_E, comm_E=prover.U.comm_W, X=prover.U.X, u=prover.U.u)
    rep = prover.check()
    assert (rep.bad_rows, rep.comm_W_ok, rep.comm_E_ok, rep.ok) == (0, False, False, False)


@pytest.mark.parametrize("fid", [O.FIELD_FQ, O.FIELD_FP])
def test_report_exactness(gpu_lib, fid):
    """Count and first row equal the oracle's for every corruption; cons = 338: three 128-thread blocks, last warp
    partial (338 % 32 = 18)."""
    shape, W, E, u, X = relaxed_instance(fid, 100, 37)
    m, cons = shape.m, shape.num_cons
    assert cons == 338
    gs = _gpu_shape(fid, shape)

    def check(W_, E_, u_):
        rep = gs.is_sat_relaxed(None, W_, E_, N.RelaxedR1CSInstance(None, None, list(X), u_))
        assert (rep.bad_rows, rep.first_bad_row) == _want(shape, W_, E_, u_, X)
        assert rep.comm_W_ok is None and rep.comm_E_ok is None
        return rep

    assert check(W, E, u).ok
    for rows in ([0], [cons - 1], [5, 130, 300], [129, 256, 337]):
        E2 = list(E)
        for r in rows:
            E2[r] = (E2[r] + 1) % m
        rep = check(W, E2, u)
        assert (rep.bad_rows, rep.first_bad_row, rep.ok) == (len(rows), rows[0], False)
    W2 = list(W)
    W2[hub_variable(shape)] = (W2[hub_variable(shape)] + 3) % m
    assert check(W2, E, u).bad_rows >= 2
    assert check(W, E, (u + 7) % m).bad_rows > cons // 2
    rep = check(W, [(e + 1) % m for e in E], u)   # every row
    assert (rep.bad_rows, rep.first_bad_row) == (cons, 0)
    assert check(W, None, u).bad_rows > 0        # E omitted from a relaxed instance


@pytest.mark.parametrize("raw", [False, True])
def test_commitments_compared_as_group_elements(gpu_lib, raw):
    fid, cid = O.FIELD_FQ, O.CURVE_PALLAS
    cv = O.CURVES[cid]
    shape, W, E, u, X = relaxed_instance(fid, 10, 100)
    gs = _gpu_shape(fid, shape)
    gens = G.Generators.progression(cid, K0, D, max(shape.num_cons, shape.num_vars), table=True, raw_jacobian=raw)
    cW, cE = cv.msm_known_dlog(W, K0, D), cv.msm_known_dlog(E, K0, D)
    rep = gs.is_sat_relaxed(gens, W, E, N.RelaxedR1CSInstance(cW, cE, list(X), u))
    assert (rep.bad_rows, rep.first_bad_row, rep.comm_W_ok, rep.comm_E_ok) == (0, None, True, True)
    # comm_E of a different vector: index 3 = 0, the rows still hold
    other = cv.msm_known_dlog([(e + 1) % shape.m for e in E], K0, D)
    rep = gs.is_sat_relaxed(gens, W, E, N.RelaxedR1CSInstance(cW, other, list(X), u))
    assert (rep.bad_rows, rep.comm_W_ok, rep.comm_E_ok, rep.ok) == (0, True, False, False)
    # the correct commitments as un-normalised Jacobian points (Z != 1)
    py = random.Random(5)
    jW, jE = (_jac_unnormalised(cv, p, py.randrange(2, cv.base)) for p in (cW, cE))
    rep = gs.is_sat_relaxed(gens, W, E, N.RelaxedR1CSInstance(jW, jE, list(X), u))
    assert (rep.comm_W_ok, rep.comm_E_ok) == (True, True)
    # a fresh instance as relaxed (u = 1, E = 0): the identity is commit(E)
    shape0, W0, X0 = fresh_instance(fid, 10, 0, 100)
    rep = gs.is_sat_relaxed(gens, W0, [0] * shape.num_cons, N.RelaxedR1CSInstance(cv.msm_known_dlog(W0, K0, D), bytes(96), list(X0), 1))
    assert (rep.bad_rows, rep.comm_W_ok, rep.comm_E_ok) == (0, True, True)
    rep = gs.is_sat_relaxed(gens, W0, [0] * shape.num_cons, N.RelaxedR1CSInstance(None, O.jac_to_bytes(cv, cE), list(X0), 1))
    assert (rep.comm_W_ok, rep.comm_E_ok) == (None, False)
    # strict is_sat: the fresh instance passes, the relaxed one passed as strict does not
    rep = gs.is_sat(gens, W0, X0, cv.msm_known_dlog(W0, K0, D))
    assert (rep.bad_rows, rep.comm_W_ok, rep.comm_E_ok, rep.ok) == (0, True, None, True)
    rep = gs.is_sat(gens, W, X, cW)
    assert rep.bad_rows == _want(shape, W, None, 1, X)[0] > 0 and rep.comm_W_ok and not rep.ok


def test_dev_counters_match_the_host_entry_point(gpu_lib):
    import torch
    fid = O.FIELD_FP
    shape, W, E, u, X = relaxed_instance(fid, 100, 37)
    m = shape.m
    gs = _gpu_shape(fid, shape)
    E2 = list(E)
    for r in (3, 200, 337):
        E2[r] = (E2[r] + 9) % m

    def dev(b):
        return torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()

    Wd, Ed, uXd = dev(O.fes_to_bytes(W, m)), dev(O.fes_to_bytes(E2, m)), dev(O.fes_to_bytes([u] + X, m))
    counts = torch.full((2,), -1, dtype=torch.int64, device="cuda")
    for E_, Edev in ((E2, Ed), (None, None)):
        gs.is_sat_relaxed_dev(Wd, Edev, uXd, counts)
        torch.cuda.synchronize()
        host = gs.is_sat_relaxed(None, W, E_, N.RelaxedR1CSInstance(None, None, list(X), u))
        got = counts.cpu().tolist()
        assert got == [host.bad_rows, shape.num_cons if host.first_bad_row is None else host.first_bad_row]
        assert host.bad_rows == len(unsat_rows(shape, W, E_, u, X))
    assert counts.cpu().tolist()[0] > 0


@pytest.mark.parametrize("fid,cid,t,aug", [(O.FIELD_FQ, O.CURVE_PALLAS, 1024, 9800), (O.FIELD_FQ, O.CURVE_PALLAS, 4096, 9800),
                                           (O.FIELD_FQ, O.CURVE_PALLAS, 16384, 9800), (O.FIELD_FP, O.CURVE_VESTA, 0, 10300)])
def test_baseline_sizes(gpu_lib, fid, cid, t, aug):
    """BASELINE config 3 sizes: one relaxed instance each, satisfied and with one E entry corrupted, commitments too.
    (The secondary block has no step rounds, so a fold of two of its fresh instances leaves E = 0: E = Az.Bz - u.Cz.)"""
    cv = O.CURVES[cid]
    shape, W, E, u, X = relaxed_instance(fid, t, aug) if t else relaxed_by_error(fid, t, aug)
    m, cons = shape.m, shape.num_cons
    assert any(E)
    gs = _gpu_shape(fid, shape)
    gens = G.Generators.progression(cid, K0, D, max(cons, shape.num_vars), table=True)
    U = N.RelaxedR1CSInstance(cv.msm_known_dlog(W, K0, D), cv.msm_known_dlog(E, K0, D), list(X), u)
    rep = gs.is_sat_relaxed(gens, W, E, U)
    assert (rep.bad_rows, rep.first_bad_row, rep.comm_W_ok, rep.comm_E_ok) == (0, None, True, True)
    bad = cons - 1 - 1000 if cons > 2000 else cons // 2
    E[bad] = (E[bad] + 1) % m
    rep = gs.is_sat_relaxed(gens, W, E, U)
    assert (rep.bad_rows, rep.first_bad_row, rep.comm_W_ok, rep.comm_E_ok) == (1, bad, True, False)
    assert unsat_rows(shape, W, E, u, X) == [bad]


def test_argument_and_state_errors(gpu_lib):
    from vdf_b200 import VdfGpuError
    lib = gpu_lib
    fid = O.FIELD_FQ
    shape, W, E, u, X = relaxed_instance(fid, 5, 0)
    m = shape.m
    gs = _gpu_shape(fid, shape)
    U = N.RelaxedR1CSInstance(None, None, list(X), u)
    n = max(shape.num_cons, shape.num_vars)
    wrong_curve = G.Generators.progression(O.CURVE_VESTA, K0, D, n)        # scalars in Fp, shape over Fq
    too_few = G.Generators.progression(O.CURVE_PALLAS, K0, D, n - 1)
    right = G.Generators.progression(O.CURVE_PALLAS, K0, D, n)
    for g in (wrong_curve, too_few):
        with pytest.raises(VdfGpuError) as e:
            gs.is_sat_relaxed(g, W, E, U)
        assert e.value.code == -1
    with pytest.raises(VdfGpuError) as e:   # comm_E without E
        gs.is_sat_relaxed(right, W, None, N.RelaxedR1CSInstance(None, bytes(96), list(X), u))
    assert e.value.code == -1
    Wb, Eb, ub, Xb = (O.fes_to_bytes(v, m) for v in (W, E, [u], X))
    assert lib.vdfgpu_r1cs_is_sat_relaxed(gs._h, None, Wb, Eb, ub, Xb, None, None, None) == -1   # null report
    rep = (ctypes.c_uint64 * 4)()
    assert lib.vdfgpu_r1cs_is_sat_relaxed(gs._h, None, Wb, Eb, ub, None, None, None, rep) == -1   # null X, io = 2
    assert lib.vdfgpu_r1cs_is_sat_relaxed(gs._h, None, Wb, Eb, ub, Xb, None, None, rep) == 0
    assert list(rep) == [0, shape.num_cons, 2, 2]
    with pytest.raises(ValueError):
        gs.is_sat_relaxed(None, W[:-1], E, U)
    with pytest.raises(ValueError):
        gs.is_sat(None, W, X[:-1])
    prover = N.RunningProver(gs, right)
    with pytest.raises(VdfGpuError) as e:
        prover.check()
    assert e.value.code == -3
    prover.close()


def test_cpp_sat_check(tmp_path):
    exe = build_sat_check(tmp_path)
    sat_check_fixtures(tmp_path)
    r = subprocess.run([str(exe), str(tmp_path)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stdout + r.stderr
