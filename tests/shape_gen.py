"""General R1CS shapes for the kernel tests (tests/test_r1cs_general_shapes.py, tests/test_gpu_r1cs_general.py), built
on the oracle.  The step shapes of oracle/pasta.py are regular: every row is short, every coefficient is non-zero, only
u's column is heavy and no constraint reads the public IO X.  The shapes here have what those lack:

  * rows of 0 to 40 entries per matrix, so a row can be empty in A and not in C;
  * columns spread over W, u and every X column;
  * coefficients 0 (written explicitly: the C ABI keeps it), 1, m - 1, 2, m - 2 and uniform values;
  * repeated (row, col) pairs;
  * one column with exactly HostCsc::HEAVY = 64 entries (the last the per-column kernel sums), one with 65 (the first
    the per-block kernel sums) and one with about 5000 (an X column when there is one, else u);
  * num_io of 0, 2 or 7.

Also a step instance whose public IO is constrained (io_bound_instance): nova's augmented circuit exposes two hash
outputs as X and constrains them; the IO-binding block below does the same through _ShapeBuilder's X ids -2, -3."""
import functools
import random
from typing import List, Tuple

from oracle import pasta as O

HEAVY = 64   # vdf_b200/csrc/r1cs_host.hpp HostCsc::HEAVY


def _coeff(py: random.Random, m: int) -> int:
    k = py.randrange(6)
    return (0, 1, m - 1, 2, m - 2)[k] if k < 5 else py.randrange(m)


def _row_len(py: random.Random) -> int:
    u = py.random()
    if u < 0.2:
        return 0
    if u < 0.75:
        return py.randint(1, 3)
    if u < 0.95:
        return py.randint(4, 10)
    return py.randint(11, 40)


@functools.lru_cache(maxsize=None)
def general_shape(fid: int, cons: int, vars_: int, io: int, seed: int = 1) -> O.R1CSShape:
    """A shape with the properties listed in the module docstring.  cons should not be a multiple of 32."""
    m = O.MODULUS[fid]
    py = random.Random(seed * 1000003 + cons * 31 + io)
    ncols = vars_ + 1 + io
    u_col, x_cols = vars_, list(range(vars_ + 1, ncols))
    col64, col65 = py.randrange(vars_ // 2), vars_ // 2 + py.randrange(vars_ // 2)
    big = x_cols[-1] if x_cols else u_col
    special = {col64, col65, big}
    mats: Tuple[List, List, List] = ([], [], [])

    def draw_col() -> int:
        while True:
            u = py.random()
            c = py.choice(x_cols) if (u < 0.12 and x_cols) else (u_col if u < 0.18 else py.randrange(vars_))
            if c not in special:
                return c

    for r in range(cons):
        for M in mats:
            row: List[Tuple[int, int, int]] = []
            for _ in range(_row_len(py)):
                c = row[py.randrange(len(row))][1] if row and py.random() < 0.1 else draw_col()   # a repeated pair
                row.append((r, c, _coeff(py, m)))
            M.extend(row)
    # the special columns: exactly 64 and 65 entries, about 5000 (rows repeat when cons < 5000)
    for c, n in ((col64, HEAVY), (col65, HEAVY + 1), (big, 5000 + py.randrange(100))):
        for _ in range(n):
            mats[py.randrange(3)].append((py.randrange(cons), c, _coeff(py, m)))
    for M in mats:
        py.shuffle(M)   # COO order is arbitrary; the CSR build is stable within a row
    return O.R1CSShape(m, cons, vars_, io, *mats)


def column_counts(shape: O.R1CSShape) -> List[int]:
    n = [0] * (shape.num_vars + 1 + shape.num_io)
    for M in (shape.A, shape.B, shape.C):
        for _, c, _ in M:
            n[c] += 1
    return n


def random_vec(py: random.Random, m: int, n: int) -> List[int]:
    """Uniform values with the edge values 0, 1 and m - 1 mixed in."""
    return [(0, 1, m - 1)[k % 3] if k % 17 == 5 else py.randrange(m) for k in range(n)]


def relaxed_instance(shape: O.R1CSShape, seed: int = 2):
    """(W, E, u, X) with random W, X, u != 1 and E := Az.Bz - u.Cz: a satisfied relaxed instance of any shape."""
    py = random.Random(seed)
    m = shape.m
    W, X = random_vec(py, m, shape.num_vars), random_vec(py, m, shape.num_io)
    u = py.randrange(2, m)
    Az, Bz, Cz = shape.multiply_vec(shape.z_of(W, u, X))
    return W, [(a * b - u * c) % m for a, b, c in zip(Az, Bz, Cz)], u, X


# ---- a step instance whose public IO is constrained --------------------------------------------------------------
def _io_value(s: O.State, m: int, salt: int) -> int:
    """Stand-in for a hash output of the step (nova exposes two Poseidon outputs as X): differs from step to step."""
    return pow((s.x + 2 * s.y + 3 * s.i + salt) % m, 5, m)


def io_bound_step(fid: int, t: int, state: O.State, aug: int):
    """(shape, W, X): make_step_instance's shape (same augmented block and step rounds) followed by an IO-binding block
    that reads X = (X0, X1) in A, B and C, next to witness variables:
        X0 * 1 = x0copy,   X1 * X0 = p,   (X1 + 2 out_x) * (X0 - out_y) = q,   (X0 + X1) * 1 = x0copy + 2 X1 - s
    with s = X1 as a witness value, so that a change of X1 alone breaks the last row too (its C part reads X).
    u = 1, E = 0 holds (a strictly satisfied fresh instance)."""
    vdf = O.MinRootVDF(fid)
    m = vdf.m
    rng = O.XorShiftRng(O.TEST_SEED)
    sb = O._ShapeBuilder(m, 2)
    if aug:
        O.synth_augmented_block(sb, rng, aug)
    zin = (sb.alloc(state.x), sb.alloc(state.y), sb.alloc(state.i))
    out = O.synth_inverse_minroot(sb, vdf, zin, t)
    X0 = _io_value(state, m, 1)
    X1 = _io_value(O.State(*(sb.values[v] for v in out)), m, 2)
    ONE, x0, x1 = sb.ONE, -2, -3
    x0copy = sb.alloc(X0)
    sb.enforce({x0: 1}, {ONE: 1}, {x0copy: 1})
    p = sb.alloc(X1 * X0)
    sb.enforce({x1: 1}, {x0: 1}, {p: 1})
    q = sb.alloc((X1 + 2 * sb.values[out[0]]) * (X0 - sb.values[out[1]]))
    sb.enforce({x1: 1, out[0]: 2}, {x0: 1, out[1]: m - 1}, {q: 1})
    s = sb.alloc(X1)
    sb.enforce({x0: 1, x1: 1}, {ONE: 1}, {x0copy: 1, x1: 2, s: m - 1})
    shape, W = sb.finish()
    return shape, W, [X0, X1]


@functools.lru_cache(maxsize=None)
def fresh_instance(fid: int, t: int, k: int, aug: int):
    """(shape, W, X): the k-th fresh IO-bound instance along the seed-42 chain (the shape is the same for every k)."""
    from tests.sat_ref import chain_state
    return io_bound_step(fid, t, chain_state(fid, t, k), aug)
