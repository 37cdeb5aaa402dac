"""CPU: the R1CS functors (r1cs.cuh: MultiplyVecFn, CrossTermFn, ScaleRowsFn + BindRowsFn + BindHeavyFn, FoldFn,
RelaxedSatFn) run by a CPU loop (tests/emul) on the general shapes of tests/shape_gen.py -- constraints that read X,
explicit zero coefficients, repeated pairs, empty and long rows, columns of exactly 64 and 65 entries, num_io 0, 2 and 7
-- against the oracle, byte for byte."""
import ctypes
import random
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import pasta as O
from tests import shape_gen as S
from tests.sat_ref import unsat_rows
from tests.util import aligned, ptr

ROOT = Path(__file__).resolve().parent.parent
SZ = ctypes.c_size_t
FIELDS = [O.FIELD_FQ, O.FIELD_FP]
# (cons, vars, io): cons % 32 != 0; io 0, 2 and 7
DIMS = [(517, 300, 0), (1337, 900, 2), (2003, 1500, 7)]


@pytest.fixture(scope="module")
def emul_sat(tmp_path_factory):
    src = ROOT / "tests" / "emul" / "emul_sat.cpp"
    lib = tmp_path_factory.mktemp("emul_sat") / "libvdf_emul_sat.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", str(lib), str(src)],
                   check=True)
    return ctypes.CDLL(str(lib))


class _Coo:
    """The shape's COO arrays as emul_r1cs / emul_r1cs_sat take them (kept alive with the object)."""

    def __init__(self, shape):
        coo = O.shape_to_coo_bytes(shape)
        self.keep = [aligned(b) for M in coo for b in M[:3]]
        self.args = []
        for k, M in enumerate(coo):
            self.args += [ptr(self.keep[3 * k]), ptr(self.keep[3 * k + 1]), ptr(self.keep[3 * k + 2]), SZ(M[3])]
        self.dims = (SZ(shape.num_cons), SZ(shape.num_vars), SZ(shape.num_io))


def _fes(v, m):
    return aligned(O.fes_to_bytes(v, m) or bytes(32))


def _r1cs(emul, fid, shape, mode, W1, u1, X1, W2=None, X2=None):
    m = shape.m
    c = _Coo(shape)
    n_out = {0: 3 * shape.num_cons, 1: shape.num_cons, 2: shape.num_vars + 1 + shape.num_io}[mode]
    out = np.zeros(n_out * 32, np.uint8)
    bufs = [_fes(W1, m), _fes(u1, m), _fes(X1, m), _fes(W2 or [0], m), _fes(X2 or [0], m)]
    rc = emul.emul_r1cs(fid, mode, *c.dims, *c.args, *[ptr(b) for b in bufs], ptr(out))
    return rc, O.fes_from_bytes(out.tobytes(), m)


@pytest.mark.parametrize("fid", FIELDS)
@pytest.mark.parametrize("cons,vars_,io", DIMS)
def test_multiply_vec_and_cross_term(emul, fid, cons, vars_, io):
    shape = S.general_shape(fid, cons, vars_, io)
    m = shape.m
    py = random.Random(cons + io)
    W1, X1, u1 = S.random_vec(py, m, vars_), S.random_vec(py, m, io), py.randrange(2, m)
    W2, X2 = S.random_vec(py, m, vars_), S.random_vec(py, m, io)
    rc, got = _r1cs(emul, fid, shape, 0, W1, [u1], X1)
    Az, Bz, Cz = shape.multiply_vec(shape.z_of(W1, u1, X1))
    assert rc == 0 and got == Az + Bz + Cz
    # X1 != X2 and u1 != 1: T depends on both IO vectors and on u1
    rc, T = _r1cs(emul, fid, shape, 1, W1, [u1], X1, W2, X2)
    assert rc == 0 and T == shape.cross_term(W1, u1, X1, W2, X2)
    if io:
        assert T != shape.cross_term(W1, u1, X1, W2, X1), "T must depend on X2"
        assert T != shape.cross_term(W1, u1, X2, W2, X2), "T must depend on X1"


@pytest.mark.parametrize("fid", FIELDS)
@pytest.mark.parametrize("cons,vars_,io", DIMS)
def test_bind_rows(emul, fid, cons, vars_, io):
    shape = S.general_shape(fid, cons, vars_, io)
    m = shape.m
    counts = S.column_counts(shape)
    assert S.HEAVY in counts and S.HEAVY + 1 in counts
    py = random.Random(7 * cons + io)
    eq = S.random_vec(py, m, cons)
    for r_abc in ([py.randrange(m) for _ in range(3)], [0, 1, m - 1]):
        heavy, got = _r1cs(emul, fid, shape, 2, eq, r_abc, [])
        assert heavy == sum(1 for n in counts if n > S.HEAVY)
        want = shape.bind_rows(eq, r_abc)
        assert got == want
        assert any(want[vars_ + 1:]) or not io


@pytest.mark.parametrize("fid", FIELDS)
def test_fold(emul, fid):
    shape = S.general_shape(fid, 1337, 900, 2)
    m = shape.m
    py = random.Random(11)
    W1, W2 = S.random_vec(py, m, 900), S.random_vec(py, m, 900)
    E1, T = S.random_vec(py, m, 1337), S.random_vec(py, m, 1337)
    for r in (py.randrange(1 << 128), m - 1, 0):
        w1, e1 = _fes(W1, m), _fes(E1, m)
        emul.emul_fold(fid, ptr(w1), ptr(_fes(W2, m)), SZ(900), ptr(e1), ptr(_fes(T, m)), SZ(1337), ptr(_fes([r], m)))
        assert O.fes_from_bytes(w1.tobytes(), m) == O.fold_vec(W1, W2, r, m)
        assert O.fes_from_bytes(e1.tobytes(), m) == O.fold_vec(E1, T, r, m)


def _sat(emul_sat, fid, shape, W, E, u, X):
    m = shape.m
    c = _Coo(shape)
    e = _fes(E, m) if E is not None else None
    out = np.zeros(2, np.uint64)
    rc = emul_sat.emul_r1cs_sat(fid, *c.dims, *c.args, ptr(_fes(W, m)), ptr(e) if e is not None else None,
                                ptr(_fes([u], m)), ptr(_fes(X, m)), ptr(out))
    assert rc == 0
    return int(out[0]), int(out[1])


def _want(shape, W, E, u, X):
    bad = unsat_rows(shape, W, E, u, X)
    return len(bad), (bad[0] if bad else shape.num_cons)


@pytest.mark.parametrize("fid", FIELDS)
@pytest.mark.parametrize("cons,vars_,io", DIMS)
def test_sat_on_general_shapes(emul_sat, fid, cons, vars_, io):
    shape = S.general_shape(fid, cons, vars_, io)
    m = shape.m
    W, E, u, X = S.relaxed_instance(shape)
    assert _sat(emul_sat, fid, shape, W, E, u, X) == (0, cons)
    E2 = list(E)
    E2[cons - 1] = (E2[cons - 1] + 1) % m
    assert _sat(emul_sat, fid, shape, W, E2, u, X) == (1, cons - 1)
    assert _sat(emul_sat, fid, shape, W, E, (u + 1) % m, X) == _want(shape, W, E, (u + 1) % m, X)
    for j in range(io):   # one X entry only: the rows that read that column, and no other
        X2 = list(X)
        X2[j] = (X2[j] + 3) % m
        want = _want(shape, W, E, u, X2)
        assert want[0] > 0
        assert _sat(emul_sat, fid, shape, W, E, u, X2) == want


@pytest.mark.parametrize("fid", FIELDS)
def test_sat_io_bound_step_instance(emul_sat, fid):
    """The strict relation on the IO-bound step instance holds; a corrupted X1 breaks exactly the IO-binding rows
    that read it."""
    shape, W, X = S.fresh_instance(fid, 5, 0, 64)
    cons = shape.num_cons
    assert _sat(emul_sat, fid, shape, W, None, 1, X) == (0, cons)
    X2 = [X[0], (X[1] + 1) % shape.m]
    want = _want(shape, W, None, 1, X2)
    assert want[0] == 3 and want[1] == cons - 3   # X1 * X0 = p, the mixed row, (X0 + X1) * 1 = x0copy + X1
    assert _sat(emul_sat, fid, shape, W, None, 1, X2) == want
