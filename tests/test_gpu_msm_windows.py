"""GPU: the Pippenger MSM at every window size c = 2..24 and on every stage-6 bucket-reduction path, with scalars that
reach each branch of the signed-digit recoding (tests/msm_cases.py), sparse and single-bucket inputs at the sizes where
the plan runs batched-affine rounds, the record-reduction variants, CUDA-graph replay with changing data, and the plain
layout at the sizes that select each of its window sizes.  Every expected value is exact: the known-discrete-log
identity over a progression P_i = (k0 + i d) G, or the oracle's MSM.

Stage 6 (msm_finish) takes, for B = 2^(c-1) buckets per set, NBT bucket sets and chunk 2^logm:
  latency  8 <= B <= 32768: bit decomposition; its pair sums by BitPairQuadFn or, above 65536 pairs, BitPairFn
  hybrid   T0 = B / 2^logm in 8..65536: one level of chunk running sums, then the same on the T0 chunk totals
  tree     anything else: recursive chunk running sums (msm_reduce_tree)
The test ids name the path each case takes (stage6() below restates the selection)."""
import ctypes
import random

import numpy as np
import pytest

from oracle import pasta as O
from tests.msm_cases import alt_sign, families, limbs, mont_table, one_digit, tile_index, tiled
from tests.util import known_dlog_scalar, nova_like_scalars, rand_scalars
from vdf_b200 import _lib
from vdf_b200 import msm as G

pytestmark = pytest.mark.gpu

CURVES = [O.CURVE_PALLAS, O.CURVE_VESTA]
K0, D = 0x1234567, 0x89ABCDEF01


def stage6(c: int, batch: int, logm: int = 3) -> str:
    B = 1 << (c - 1)
    if 8 <= B <= 32768:
        return "latency-quad" if batch * (c - 1) * (B // 4) <= 65536 else "latency-bitpair"
    T0 = B >> logm
    if B % (1 << logm) == 0 and 8 <= T0 <= 65536:
        nbits = T0.bit_length() - 1
        return "hybrid-quad" if batch * nbits * (T0 // 4) <= 65536 else "hybrid-plain"
    return "tree"


@pytest.fixture(scope="module", autouse=True)
def _trim(gpu_lib):
    yield
    _lib.check(gpu_lib.vdfgpu_trim())   # bucket arrays of c = 24 with batch 4 are 4 GB


def _want(cv, sc, k0=K0, d=D) -> bytes:
    return O.jac_to_bytes(cv, cv.msm_known_dlog(sc, k0, d))


def _mul_gen(cv, s: int) -> bytes:
    return O.jac_to_bytes(cv, cv.mul(s % cv.order, cv.gen))


def _batch_dev(lib, g, vecs, order):
    """vdfgpu_msm_batch_dev over device copies of `vecs`; the results as affine points (None = identity)."""
    import torch
    k = len(vecs)
    dev = [torch.frombuffer(bytearray(O.fes_to_bytes(v, order) or bytes(32)), dtype=torch.uint8).cuda() for v in vecs]
    ptrs = (ctypes.c_void_p * k)(*[t.data_ptr() for t in dev])
    lens = (ctypes.c_size_t * k)(*[len(v) for v in vecs])
    out = torch.zeros(96 * k, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    _lib.check(lib.vdfgpu_msm_batch_dev(g._h, ptrs, lens, k, out.data_ptr()))
    _lib.check(lib.vdfgpu_synchronize())
    raw = out.cpu().numpy().tobytes()
    return [raw[96 * j:96 * j + 96] for j in range(k)]


# ---- a. every window size, batch 1 and batch 4 ----------------------------------------------------------------
@pytest.mark.parametrize("cid", CURVES)
@pytest.mark.parametrize("c", [pytest.param(c, id=f"c{c}-{stage6(c, 1)}-batch4-{stage6(c, 4)}") for c in range(2, 25)])
def test_window_matrix(gpu_lib, c, cid):
    cv = O.CURVES[cid]
    n, B = 1000, 1 << (c - 1)
    g = G.Generators.progression(cid, K0, D, n, table=True, window_bits=c)
    assert g.window_bits(n) == c
    sc = tiled(c, cv.order, n, seed=c)
    assert g.commit_bytes(O.fes_to_bytes(sc, cv.order)) == _want(cv, sc)
    vecs = [sc, [one_digit(c, B)] * (n - 1), [families(c, cv.order)["zero_with_carry"]], []]
    got = _batch_dev(gpu_lib, g, vecs, cv.order)
    for j, v in enumerate(vecs):
        assert O.jac_from_bytes(cv, got[j]) == cv.msm_known_dlog(v, K0, D), (c, j)
    g.close()


# ---- b. logm moves the hybrid / tree boundary ----------------------------------------------------------------
@pytest.mark.parametrize("logm", [1, 8])
@pytest.mark.parametrize("c", [17, 20, 21, 24])
def test_window_logm(gpu_lib, c, logm, monkeypatch):
    monkeypatch.setenv("VDFGPU_MSM_LOGM", str(logm))
    want_path = {(17, 1): "hybrid", (20, 1): "tree", (21, 1): "tree", (24, 1): "tree"}.get((c, logm), "hybrid")
    assert stage6(c, 1, logm).startswith(want_path)
    n = 1000
    for cid in CURVES:
        cv = O.CURVES[cid]
        g = G.Generators.progression(cid, K0, D, n, table=True, window_bits=c)
        assert g.window_bits(n) == c
        sc = tiled(c, cv.order, n, seed=100 + c)
        assert g.commit_bytes(O.fes_to_bytes(sc, cv.order)) == _want(cv, sc), (c, logm, cid)
        g.close()


# ---- c. affine rounds where most bucket segments hold 0 or 1 entries ------------------------------------------
@pytest.mark.parametrize("c", [2, 13, 17, 24])
def test_affine_rounds_sparse_buckets(gpu_lib, c, monkeypatch):
    cid = CURVES[c % 2]
    cv = O.CURVES[cid]
    n = 1000
    g = G.Generators.progression(cid, K0, D, n, table=True, window_bits=c)
    assert g.window_bits(n) == c
    sc = tiled(c, cv.order, n, seed=200 + c)
    sb, want = O.fes_to_bytes(sc, cv.order), _want(cv, sc)
    single = O.fes_to_bytes([one_digit(c, 1)], cv.order)
    for rounds in (1, 3):
        for K in (1, 32):
            monkeypatch.setenv("VDFGPU_MSM_AFFINE", str(rounds))
            monkeypatch.setenv("VDFGPU_MSM_AFFINE_K", str(K))
            assert g.affine_rounds(n) == rounds
            assert g.commit_bytes(sb) == want, (c, rounds, K)
            assert g.commit_bytes(sb[:32 * 7]) == _want(cv, sc[:7]), (c, rounds, K)
            assert g.commit_bytes(single) == _want(cv, [one_digit(c, 1)]), (c, rounds, K)
    g.close()


# ---- d. record reduction: RecRunsFn levels, serial levels, RecBucketFn ----------------------------------------
@pytest.fixture(scope="module")
def gens_2_16(gpu_lib):
    g = G.Generators.progression(O.CURVE_PALLAS, K0, D, 1 << 16, table=True)
    yield g
    g.close()


@pytest.mark.parametrize("recbucket", ["0", "1"])
@pytest.mark.parametrize("S", ["1", "3", None])
def test_record_paths(gens_2_16, S, recbucket, monkeypatch):
    """S = 1 cuts every bucket into as many records as it has entries: RecRunsFn blocks that are one run of 256,
    several launch levels, serial RecLevelFn levels above 2^19 records, and for RecBucketFn buckets of far more than
    24 pieces (its whole-warp branch)."""
    if S is not None:
        monkeypatch.setenv("VDFGPU_MSM_S", S)
    monkeypatch.setenv("VDFGPU_MSM_RECBUCKET", recbucket)
    cv, g, n = O.PALLAS, gens_2_16, 1 << 16
    c = 15
    B = 1 << (c - 1)
    assert g.window_bits(n) == c and g.affine_rounds(n) == 0
    digits = [one_digit(c, d) for d in (1, B - 1, B)]
    sc = [digits[i * 3 // n] for i in range(n)]
    assert g.commit_bytes(O.fes_to_bytes(sc, cv.order)) == _want(cv, sc)
    py, rng = random.Random(5), O.XorShiftRng()
    sc = nova_like_scalars(py, rng, cv.order, n)
    assert g.commit_bytes(O.fes_to_bytes(sc, cv.order)) == _want(cv, sc)


# ---- e, f. one bucket, and empty or nearly empty inputs, at the sizes where the plan runs affine rounds ----------
@pytest.fixture(scope="module")
def big_gens(gpu_lib):
    sets = {}

    def get(log2n):
        if log2n not in sets:
            sets[log2n] = G.Generators.progression(O.CURVE_PALLAS, K0, D, 1 << log2n, table=True)
        return sets[log2n]
    yield get
    for g in sets.values():
        g.close()


def _progression_sum(n: int, k0: int = K0, d: int = D) -> int:
    return n * k0 + d * n * (n - 1) // 2


@pytest.mark.parametrize("log2n,c", [(20, 19), (22, 20)])
def test_one_bucket_at_scale(big_gens, log2n, c, monkeypatch):
    """Every scalar is one_digit(B): all K * n entries land in bucket B, and the plan's own affine rounds halve one
    giant segment."""
    cv, g, n = O.PALLAS, big_gens(log2n), 1 << log2n
    B = 1 << (c - 1)
    assert g.window_bits(n) == c and g.affine_rounds(n) > 0
    s = one_digit(c, B)
    sb = O.fes_to_bytes([s], cv.order) * n
    want = _mul_gen(cv, s * _progression_sum(n))
    assert g.commit_bytes(sb) == want
    if log2n == 20:
        # short ranges: more than 2^19 records in long runs, so the serial RecLevelFn levels run first
        monkeypatch.setenv("VDFGPU_MSM_S", "4")
        assert g.commit_bytes(sb) == want


def test_one_bucket_equal_generators(gpu_lib):
    """All generators equal (progression with d = 0) and scalars one_digit(d) / alt_sign(d): bucket d holds
    2^(c w) P and -2^(c w) P, so equal points and opposite points meet in the affine rounds."""
    cv, n, c = O.PALLAS, 1 << 20, 19
    d = (1 << (c - 1)) - 1
    k0 = 0x5EED
    g = G.Generators.progression(cv.cid, k0, 0, n, table=True)
    assert g.window_bits(n) == c and g.affine_rounds(n) > 0
    a, b = one_digit(c, d), alt_sign(c, d)
    sb = O.fes_to_bytes([a, b], cv.order) * (n // 2)
    assert g.commit_bytes(sb) == _mul_gen(cv, (a + b) * (n // 2) * k0)
    g.close()


@pytest.mark.parametrize("log2n,c", [(20, 19), (22, 20)])
def test_empty_and_last_only_at_scale(big_gens, log2n, c):
    cv, g, n = O.PALLAS, big_gens(log2n), 1 << log2n
    assert g.window_bits(n) == c and g.affine_rounds(n) > 0
    assert g.commit_bytes(bytes(32 * n)) == bytes(96)
    for s in (1, families(c, cv.order)["zero_with_carry"], cv.order - 1):
        sb = bytearray(32 * n)
        sb[-32:] = O.fe_to_bytes(s, cv.order)
        assert g.commit_bytes(bytes(sb)) == _mul_gen(cv, s * (K0 + (n - 1) * D)), s


# ---- g. graph replay of one plan with changing data ----------------------------------------------------------
def test_graph_replay_changing_data(gpu_lib):
    cv, n = O.VESTA, 1 << 14
    g = G.Generators.progression(cv.cid, K0, D, n, table=True)
    c = g.window_bits(n)
    assert c == 13
    B = 1 << (c - 1)
    rng, py = O.XorShiftRng(), random.Random(31)
    uni = rand_scalars(rng, cv.order, n)
    fam = families(c, cv.order)
    seq = [uni, [0] * n, [one_digit(c, B)] * n, [fam["zero_with_carry"]] * n, nova_like_scalars(py, rng, cv.order, n),
           uni, uni[:n - 1], uni]
    for k, sc in enumerate(seq):
        assert g.commit_bytes(O.fes_to_bytes(sc, cv.order)) == _want(cv, sc), k
    g.close()


# ---- h. plain layout at the sizes that select each of its window sizes -------------------------------------------
@pytest.mark.parametrize("log2n,c,rounds", [(13, 7, 0), (15, 9, 0), (17, 13, 0), (22, 16, 3), (23, 17, None)])
def test_plain_layout_window_sizes(gpu_lib, log2n, c, rounds):
    """A plain set picks c from n on every call; W bucket sets, the FinalFn Horner over the windows."""
    cid = CURVES[log2n % 2]
    cv, n = O.CURVES[cid], 1 << log2n
    g = G.Generators.progression(cid, K0, D, n)
    assert g.window_bits(n) == c
    if rounds is not None:
        assert g.affine_rounds(n) == rounds
    vals = list(families(c, cv.order).values()) + rand_scalars(O.XorShiftRng(), cv.order, 64)
    idx = tile_index(n, len(vals), seed=log2n)
    sb = mont_table(vals, cv.order)[idx].tobytes()
    acc = known_dlog_scalar(limbs(vals)[idx], K0, D)
    assert g.commit_bytes(sb) == _mul_gen(cv, acc)
    g.close()


# ---- i. pasta-msm's one-shot symbol with raw (non-Montgomery) scalars ---------------------------------------------
@pytest.mark.parametrize("cid", CURVES)
def test_mult_pippenger_raw_families(gpu_lib, cid):
    cv = O.CURVES[cid]
    n, k0, d = 600, 3, 7
    pb = O.affines_to_bytes(cv, cv.progression(k0, d, n))
    for c in (4, 9, 16):
        sc = tiled(c, cv.order, n, seed=300 + c)
        want = _want(cv, sc, k0, d)
        assert G.mult_pippenger(cid, pb, b"".join(s.to_bytes(32, "little") for s in sc), False) == want, c
        assert G.mult_pippenger(cid, pb, O.fes_to_bytes(sc, cv.order), True) == want, c
