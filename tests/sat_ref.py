"""Reference side of the satisfiability tests (tests/test_r1cs_sat.py, tests/test_gpu_r1cs_sat.py): the violating
rows of a relaxed R1CS instance, restated from the definition on top of the oracle's multiply_vec, and the relaxed
instances the tests corrupt."""
import functools
import struct
import subprocess
from pathlib import Path
from typing import List, Optional, Sequence

from oracle import pasta as O


def unsat_rows(shape: O.R1CSShape, W: Sequence[int], E: Optional[Sequence[int]], u: int, X: Sequence[int]) -> List[int]:
    """Rows where Az.Bz != u.Cz + E (E None: E = 0): what RelaxedR1CSShape::is_sat_relaxed rejects."""
    Az, Bz, Cz = shape.multiply_vec(shape.z_of(W, u, X))
    E = [0] * shape.num_cons if E is None else E
    m = shape.m
    return [r for r, (a, b, c, e) in enumerate(zip(Az, Bz, Cz, E)) if (a * b - u * c - e) % m]


@functools.lru_cache(maxsize=None)
def chain_state(fid: int, t: int, k: int) -> O.State:
    """State of the seed-42 chain after k + 1 segments of t rounds (the slow fifth-root direction, oracle)."""
    ovdf = O.MinRootVDF(fid)
    if k < 0:
        return O.State(O.field_random(O.XorShiftRng(), ovdf.m), 0, 1)
    return ovdf.eval(chain_state(fid, t, k - 1), t)


def fresh_instance(fid: int, t: int, k: int, aug: int):
    """(shape, W, X): the k-th fresh instance of the step shape."""
    shape, W, X, _ = O.make_step_instance(fid, t, chain_state(fid, t, k), aug_cons=aug)
    return shape, W, X


R0 = 0x1F2E3D4C5B6A79880123456789ABCDEF


def relaxed_instance(fid: int, t: int, aug: int):
    """(shape, W, E, u, X): fresh instance 1 folded into fresh instance 0 by the oracle (u != 1, E != 0)."""
    shape, W0, X0 = fresh_instance(fid, t, 0, aug)
    _, W1, X1 = fresh_instance(fid, t, 1, aug)
    m = shape.m
    T = shape.cross_term(W0, 1, X0, W1, X1)
    W, E = O.fold_vec(W0, W1, R0, m), O.fold_vec([0] * shape.num_cons, T, R0, m)
    return shape, W, E, (1 + R0) % m, [(a + R0 * b) % m for a, b in zip(X0, X1)]


def relaxed_by_error(fid: int, t: int, aug: int, u: int = R0):
    """(shape, W, E, u, X): fresh instance 0 with u != 1 and the error vector E = Az.Bz - u.Cz that makes it hold.
    For shapes where two fresh instances barely differ (t = 0: only the augmented block, which every instance shares)
    a fold leaves E = 0; this gives a dense E instead."""
    shape, W, X = fresh_instance(fid, t, 0, aug)
    m = shape.m
    Az, Bz, Cz = shape.multiply_vec(shape.z_of(W, u, X))
    return shape, W, [(a * b - u * c) % m for a, b, c in zip(Az, Bz, Cz)], u % m, X


SAT_K0, SAT_D = 21, 5   # generators of the C++ check program: P_i = (SAT_K0 + i SAT_D) G on Pallas


def build_sat_check(out_dir: Path) -> Path:
    """tests/cpp/sat_check.cpp (the C++ host layer's satisfiability checks) linked against libvdfgpu.so."""
    from vdf_b200 import _lib
    _lib.load()
    root = Path(__file__).resolve().parent.parent
    exe = Path(out_dir) / "sat_check"
    libdir = root / "vdf_b200" / "lib"
    subprocess.run(["g++", "-O1", "-std=c++17", "-o", str(exe), str(root / "tests" / "cpp" / "sat_check.cpp"),
                    f"-L{libdir}", "-lvdfgpu", f"-Wl,-rpath,{libdir}"], check=True)
    return exe


def sat_check_fixtures(d: Path) -> None:
    """Inputs and oracle answers of sat_check: a relaxed Pallas-side instance (t = 7, 40 extra constraints), its
    commitments, and the exact reports for the instance as it is and with E[cons / 3] corrupted."""
    d = Path(d)
    fid, cv = O.FIELD_FQ, O.PALLAS
    shape, W, E, u, X = relaxed_instance(fid, 7, 40)
    m, cons = shape.m, shape.num_cons
    coo = O.shape_to_coo_bytes(shape)
    (d / "dims.bin").write_bytes(struct.pack("<6Q", cons, shape.num_vars, shape.num_io, *[c[3] for c in coo]))
    for name, (rows, cols, vals, _) in zip("abc", coo):
        (d / f"{name}_rows.bin").write_bytes(rows)
        (d / f"{name}_cols.bin").write_bytes(cols)
        (d / f"{name}_vals.bin").write_bytes(vals)
    bad = cons // 3
    E_bad = list(E)
    E_bad[bad] = (E_bad[bad] + 1) % m
    for name, v in (("W", W), ("E", E), ("E_bad", E_bad), ("u", [u]), ("X", X)):
        (d / f"{name}.bin").write_bytes(O.fes_to_bytes(v, m))
    (d / "k0_d.bin").write_bytes(SAT_K0.to_bytes(32, "little") + SAT_D.to_bytes(32, "little"))
    comm = [cv.msm_known_dlog(v, SAT_K0, SAT_D) for v in (W, E)]
    (d / "comm.bin").write_bytes(b"".join(O.jac_to_bytes(cv, p) for p in comm))
    (d / "reports.bin").write_bytes(struct.pack("<8Q", 0, cons, 1, 1, 1, bad, 1, 0))


def hub_variable(shape: O.R1CSShape) -> int:
    """The witness variable that appears in the most constraint rows."""
    rows = {}
    for M in (shape.A, shape.B, shape.C):
        for r, c, _ in M:
            if c < shape.num_vars:
                rows.setdefault(c, set()).add(r)
    return max(rows, key=lambda c: len(rows[c]))
