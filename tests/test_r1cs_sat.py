"""CPU: the satisfiability functor (r1cs.cuh RelaxedSatFn, the row part of RecursiveSNARK::verify's is_sat_relaxed /
is_sat) run by a CPU loop (tests/emul/emul_sat.cpp) against the violating rows the oracle finds; and the C++ check
program of tests/cpp/sat_check.cpp builds and fails loudly without a GPU."""
import ctypes
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import pasta as O
from tests.sat_ref import (build_sat_check, fresh_instance, hub_variable, relaxed_instance, sat_check_fixtures,
                           unsat_rows)
from tests.util import aligned, ptr

ROOT = Path(__file__).resolve().parent.parent
SZ = ctypes.c_size_t


@pytest.fixture(scope="module")
def emul_sat(tmp_path_factory):
    src = ROOT / "tests" / "emul" / "emul_sat.cpp"
    lib = tmp_path_factory.mktemp("emul_sat") / "libvdf_emul_sat.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", str(lib), str(src)],
                   check=True)
    return ctypes.CDLL(str(lib))


def _emul_counts(emul_sat, fid, shape, W, E, u, X):
    m = shape.m
    coo = O.shape_to_coo_bytes(shape)
    keep = [aligned(b) for M in coo for b in M[:3]]
    args = []
    for k, M in enumerate(coo):
        args += [ptr(keep[3 * k]), ptr(keep[3 * k + 1]), ptr(keep[3 * k + 2]), SZ(M[3])]
    w, x, uu = aligned(O.fes_to_bytes(W, m)), aligned(O.fes_to_bytes(X, m)), aligned(O.fe_to_bytes(u, m))
    e = aligned(O.fes_to_bytes(E, m)) if E is not None else None
    out = np.zeros(2, np.uint64)
    rc = emul_sat.emul_r1cs_sat(fid, SZ(shape.num_cons), SZ(shape.num_vars), SZ(shape.num_io), *args, ptr(w),
                                ptr(e) if e is not None else None, ptr(uu), ptr(x), ptr(out))
    assert rc == 0
    return int(out[0]), int(out[1])


def _want(shape, W, E, u, X):
    bad = unsat_rows(shape, W, E, u, X)
    return len(bad), (bad[0] if bad else shape.num_cons)


# aug chosen so that cons = 3t + 1 + aug is not a multiple of 32 (a partial last warp on the device)
@pytest.mark.parametrize("fid", [O.FIELD_FQ, O.FIELD_FP])
@pytest.mark.parametrize("t,aug", [(5, 0), (10, 0), (100, 37)])
def test_emulated_sat_matches_oracle(emul_sat, fid, t, aug):
    shape, W, E, u, X = relaxed_instance(fid, t, aug)
    m, cons = shape.m, shape.num_cons
    assert cons % 32 != 0 and u != 1 and any(E)
    check = lambda W_, E_, u_: _emul_counts(emul_sat, fid, shape, W_, E_, u_, X) == _want(shape, W_, E_, u_, X)  # noqa: E731
    # satisfied relaxed instance
    assert unsat_rows(shape, W, E, u, X) == []
    assert _emul_counts(emul_sat, fid, shape, W, E, u, X) == (0, cons)
    # one corrupted E entry: first row, last row, a middle row
    for row in (0, cons - 1, cons // 2):
        E2 = list(E)
        E2[row] = (E2[row] + 1) % m
        assert _emul_counts(emul_sat, fid, shape, W, E2, u, X) == (1, row)
    # a witness variable that feeds many rows
    W2 = list(W)
    hub = hub_variable(shape)
    W2[hub] = (W2[hub] + 5) % m
    assert len(unsat_rows(shape, W2, E, u, X)) >= 2
    assert check(W2, E, u)
    # a wrong u breaks every row whose constant or C part it scales
    assert len(unsat_rows(shape, W, E, (u + 1) % m, X)) > cons // 2
    assert check(W, E, (u + 1) % m)
    # E omitted from a relaxed instance (E != 0 on most rows)
    assert check(W, None, u)
    assert _emul_counts(emul_sat, fid, shape, W, None, u, X)[0] > 0
    # a fresh instance under the strict check (u = 1, E = 0)
    shape0, W0, X0 = fresh_instance(fid, t, 0, aug)
    assert _emul_counts(emul_sat, fid, shape0, W0, None, 1, X0) == (0, cons)


def test_sat_check_program_builds_and_has_no_cpu_fallback(tmp_path):
    import torch
    exe = build_sat_check(tmp_path)
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu test")
    sat_check_fixtures(tmp_path)
    r = subprocess.run([str(exe), str(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 3 and "no CPU fallback" in r.stderr, r.stdout + r.stderr
