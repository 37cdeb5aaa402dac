"""GPU parity for the Pippenger MSM (SURVEY 8a row a4) through the C ABI: bit-exact canonical points
against the Python oracle at small sizes, the known-discrete-log identity at BASELINE sizes, linearity,
edge cases (empty, zeros, identity points, duplicates, P and -P, non-Montgomery scalars)."""
import random

import pytest

from oracle import pasta as O
from vdf_b200 import msm as G
from vdf_b200.encoding import CURVE_BASE
from tests.util import nova_like_scalars, rand_scalars

pytestmark = pytest.mark.gpu

CURVES = [O.CURVE_PALLAS, O.CURVE_VESTA]


@pytest.mark.parametrize("cid", CURVES)
def test_progression_matches_oracle(gpu_lib, cid):
    cv = O.CURVES[cid]
    g = G.Generators.progression(cid, 7, 3, 100)
    assert g.export() == cv.progression(7, 3, 100)
    assert all(cv.on_curve(p) for p in g.export())
    g2 = G.Generators.progression(cid, 0, 5, 40)  # starts at the identity
    assert g2.export() == cv.progression(0, 5, 40)


@pytest.mark.parametrize("cid", CURVES)
@pytest.mark.parametrize("table", [False, True])
def test_msm_small_vs_oracle(gpu_lib, cid, table):
    cv = O.CURVES[cid]
    rng = O.XorShiftRng()
    n = 700
    pts = cv.progression(5, 11, n)
    sc = rand_scalars(rng, cv.order, n)
    sc[0], sc[1], sc[2], sc[3] = 0, 1, cv.order - 1, 1 << 128
    pts[7] = None                       # identity generator
    pts[9], sc[9] = pts[8], sc[8]       # duplicate point, same scalar (doubling inside a bucket)
    pts[11], sc[11] = cv.neg(pts[10]), sc[10]  # P and -P cancel
    want = O.jac_to_bytes(cv, cv.msm(sc, pts))
    for wb in ((0, 5, 9, 13) if table else (0,)):   # a plain set picks c from n and ignores window_bits
        g = G.Generators.from_points(cid, pts, table=table, window_bits=wb)
        assert g.commit_bytes(O.fes_to_bytes(sc, cv.order)) == want, (cid, table, wb)
        # prefix commits (nova commits to vectors shorter than the generator set)
        for k in (0, 1, 2, 33, 699):
            assert g.commit_bytes(O.fes_to_bytes(sc[:k], cv.order)) == O.jac_to_bytes(cv, cv.msm(sc[:k], pts[:k]))
        g.close()


@pytest.mark.parametrize("cid", CURVES)
def test_mult_pippenger_abi(gpu_lib, cid):
    """pasta-msm's symbol: points travel with the call; is_mont both ways."""
    cv = O.CURVES[cid]
    rng = O.XorShiftRng()
    n = 300
    pts = cv.progression(3, 7, n)
    sc = rand_scalars(rng, cv.order, n)
    want = O.jac_to_bytes(cv, cv.msm(sc, pts))
    pb = O.affines_to_bytes(cv, pts)
    assert G.mult_pippenger(cid, pb, O.fes_to_bytes(sc, cv.order), True) == want
    assert G.mult_pippenger(cid, pb, b"".join(s.to_bytes(32, "little") for s in sc), False) == want
    assert G.mult_pippenger(cid, b"", b"", True) == bytes(96)


@pytest.mark.parametrize("table", [False, True])
def test_msm_nova_like_scalars(gpu_lib, table):
    """Witness-like digits (many 0/1/small): one bucket gets ~n/4 entries -> exercises the record levels."""
    cv = O.PALLAS
    rng, py = O.XorShiftRng(), random.Random(5)
    n = 1 << 14
    k0, d = 12345, 678
    sc = nova_like_scalars(py, rng, cv.order, n)
    g = G.Generators.progression(cv.cid, k0, d, n, table=table)
    assert g.commit(sc) == cv.msm_known_dlog(sc, k0, d)


@pytest.mark.parametrize("cid", CURVES)
@pytest.mark.parametrize("table,log2n", [(False, 16), (True, 16), (False, 20), (True, 20)])
def test_msm_known_dlog_large(gpu_lib, cid, table, log2n):
    """BASELINE config 2 sizes: P_i = (k0 + i d) G  =>  MSM = (sum s_i (k0 + i d)) G, checked in O(n)."""
    cv = O.CURVES[cid]
    n = 1 << log2n
    k0, d = 0x1234567, 0x89ABCDEF01
    py = random.Random(log2n * 7 + cid)
    sc = [py.randrange(cv.order) for _ in range(n)]
    g = G.Generators.progression(cid, k0, d, n, table=table)
    got = g.commit(sc)
    assert got == cv.msm_known_dlog(sc, k0, d)
    # linearity: MSM(s + s') = MSM(s) + MSM(s')
    sc2 = [py.randrange(cv.order) for _ in range(n)]
    got2 = g.commit(sc2)
    got12 = g.commit([(a + b) % cv.order for a, b in zip(sc, sc2)])
    assert got12 == cv.add(got, got2)
    g.close()


def test_msm_known_dlog_2_22(gpu_lib):
    """The benchmark's own size (BASELINE config 2 maximum, 2^22 points, table layout c = 20): known-discrete-log
    identity, plus the same scalars through the plain layout and pasta-msm's one-shot symbol on a 2^16 prefix."""
    import numpy as np
    cv = O.PALLAS
    n = 1 << 22
    k0, d = 0x1234567, 0x89ABCDEF01
    rs = np.random.RandomState(7)
    raw = rs.randint(0, 1 << 32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
    raw[:, 7] &= 0x3FFFFFFF                                   # < 2^254: valid Montgomery-form limbs
    sb = raw.tobytes()
    g = G.Generators.progression(cv.cid, k0, d, n, table=True)
    got = O.jac_from_bytes(cv, g.commit_bytes(sb))
    # scalar value = limbs * R^-1: fold R^-1 out once instead of per element
    rinv = pow(1 << 256, -1, cv.order)
    acc = 0
    for i in range(n):
        acc += int.from_bytes(sb[32 * i:32 * i + 32], "little") * (k0 + i * d)
    assert got == cv.mul(acc * rinv % cv.order, cv.gen)
    m = 1 << 16
    want_prefix = g.commit_bytes(sb[:32 * m])
    gp = G.Generators.progression(cv.cid, k0, d, m, table=False)
    assert gp.commit_bytes(sb[:32 * m]) == want_prefix
    pts72 = bytearray(72 * m)
    from vdf_b200 import _lib
    _lib.check(gpu_lib.vdfgpu_gens_export(gp._h, 0, m, _lib.as_ptr(pts72)))
    assert G.mult_pippenger(cv.cid, bytes(pts72), sb[:32 * m], True) == want_prefix


def test_point_sum_and_sharded_combine(gpu_lib):
    """Multi-GPU path emulated as G point-range slices on one GPU (SURVEY section 4): partials combined with
    vdfgpu_point_sum equal the single-range result."""
    cv = O.PALLAS
    n, world = 1 << 12, 4
    k0, d = 99, 5
    py = random.Random(3)
    sc = [py.randrange(cv.order) for _ in range(n)]
    full = G.Generators.progression(cv.cid, k0, d, n)
    want = full.commit_bytes(O.fes_to_bytes(sc, cv.order))
    parts = []
    per = n // world
    for r in range(world):
        shard = G.Generators.progression(cv.cid, k0 + r * per * d, d, per, table=True)
        parts.append(shard.commit_bytes(O.fes_to_bytes(sc[r * per:(r + 1) * per], cv.order)))
    assert G.point_sum(cv.cid, b"".join(parts)) == want
    assert G.point_sum(cv.cid, b"") == bytes(96)
    assert O.jac_from_bytes(cv, want) == cv.msm_known_dlog(sc, k0, d)


def test_msm_argument_errors(gpu_lib):
    from vdf_b200 import VdfGpuError
    g = G.Generators.progression(0, 1, 1, 16)
    with pytest.raises(VdfGpuError):
        g.commit_bytes(bytes(32 * 17))  # more scalars than generators
    with pytest.raises(VdfGpuError):
        G.Generators.from_affine_bytes(0, b"", table=False)


@pytest.mark.parametrize("affine", ["0", "2"])
def test_msm_batch_dev(gpu_lib, affine, monkeypatch):
    """vdfgpu_msm_batch_dev: three scalar vectors of different lengths, one pass, device pointers (also with the
    batched-affine halving rounds forced on at this small size)."""
    monkeypatch.setenv("VDFGPU_MSM_AFFINE", affine)
    import ctypes

    import torch

    from vdf_b200 import _lib
    cv = O.PALLAS
    rng, py = O.XorShiftRng(), random.Random(4)
    n, k0, d = 5000, 17, 29
    g = G.Generators.progression(cv.cid, k0, d, n, table=True)
    vecs = [rand_scalars(rng, cv.order, 5000), nova_like_scalars(py, rng, cv.order, 3777), [7]]
    dev = [torch.frombuffer(bytearray(O.fes_to_bytes(v, cv.order)), dtype=torch.uint8).cuda() for v in vecs]
    ptrs = (ctypes.c_void_p * 3)(*[t.data_ptr() for t in dev])
    lens = (ctypes.c_size_t * 3)(*[len(v) for v in vecs])
    out = torch.zeros(96 * 3, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    _lib.check(gpu_lib.vdfgpu_msm_batch_dev(g._h, ptrs, lens, 3, out.data_ptr()))
    _lib.check(gpu_lib.vdfgpu_synchronize())
    raw = out.cpu().numpy().tobytes()
    for j, v in enumerate(vecs):
        assert O.jac_from_bytes(cv, raw[96 * j:96 * j + 96]) == cv.msm_known_dlog(v, k0, d)


@pytest.mark.parametrize("table", [False, True])
def test_msm_host_chunked_overlap(gpu_lib, table, monkeypatch):
    """vdfgpu_msm's chunked schedule (H2D of chunk k+1 under the accumulation of chunk k, one bucket array):
    forced on a small input, ragged last chunk, identical bytes to the single-pass result."""
    cv = O.PALLAS
    rng, py = O.XorShiftRng(), random.Random(8)
    n, k0, d = 5001, 3, 7
    sc = nova_like_scalars(py, rng, cv.order, n)
    g = G.Generators.progression(cv.cid, k0, d, n, table=table)
    sb = O.fes_to_bytes(sc, cv.order)
    monkeypatch.setenv("VDFGPU_MSM_CHUNKS", "1")
    single = g.commit_bytes(sb)
    for chunks in ("2", "4", "7"):
        monkeypatch.setenv("VDFGPU_MSM_CHUNKS", chunks)
        assert g.commit_bytes(sb) == single
    monkeypatch.setenv("VDFGPU_MSM_AFFINE", "2")   # chunks + batched-affine halving rounds
    assert g.commit_bytes(sb) == single
    assert O.jac_from_bytes(cv, single) == cv.msm_known_dlog(sc, k0, d)


@pytest.mark.parametrize("cid", CURVES)
@pytest.mark.parametrize("table", [False, True])
def test_msm_affine_rounds(gpu_lib, cid, table, monkeypatch):
    """Optional batched-affine halving rounds in front of the XYZZ accumulation (msm_affine.cuh, off by default):
    identical bytes for any number of rounds, on uniform and Nova-like scalars and on exceptional pairs."""
    cv = O.CURVES[cid]
    rng, py = O.XorShiftRng(), random.Random(11 + cid)
    n, k0, d = 1 << 16, 5, 9
    g = G.Generators.progression(cid, k0, d, n, table=table, window_bits=9)   # ~250+ entries per bucket
    uni = O.fes_to_bytes([py.randrange(cv.order) for _ in range(n)], cv.order)
    skew_sc = nova_like_scalars(py, rng, cv.order, n)
    skew = O.fes_to_bytes(skew_sc, cv.order)
    monkeypatch.setenv("VDFGPU_MSM_AFFINE", "0")
    want_uni, want_skew = g.commit_bytes(uni), g.commit_bytes(skew)
    assert O.jac_from_bytes(cv, want_skew) == cv.msm_known_dlog(skew_sc, k0, d)
    for rounds, K in (("1", "64"), ("3", "7"), ("5", "32")):
        monkeypatch.setenv("VDFGPU_MSM_AFFINE", rounds)
        monkeypatch.setenv("VDFGPU_MSM_AFFINE_K", K)
        assert g.commit_bytes(uni) == want_uni, (rounds, K)
        assert g.commit_bytes(skew) == want_skew, (rounds, K)
    g.close()
    # equal points (doublings in every round), P + (-P), identity generators
    m = 2000
    pts = cv.progression(3, 1, 8) * (m // 8)
    pts[5] = None
    for k in range(16, 64, 2):
        pts[k + 1] = cv.neg(pts[k])
    sc = [12345] * m
    g = G.Generators.from_points(cid, pts, table=table, window_bits=6)
    monkeypatch.setenv("VDFGPU_MSM_AFFINE", "0")
    want = g.commit_bytes(O.fes_to_bytes(sc, cv.order))
    assert want == O.jac_to_bytes(cv, cv.msm(sc, pts))
    monkeypatch.setenv("VDFGPU_MSM_AFFINE", "4")
    monkeypatch.setenv("VDFGPU_MSM_AFFINE_K", "8")
    assert g.commit_bytes(O.fes_to_bytes(sc, cv.order)) == want
    g.close()


@pytest.mark.parametrize("cid", CURVES)
def test_raw_jacobian_output(gpu_lib, cid):
    """VDFGPU_GENS_RAW_JACOBIAN: the un-normalised (X, Y, Z) result is the same group element (what pasta-msm returns
    is un-normalised too); identity stays (0, 0, 0)."""
    cv = O.CURVES[cid]
    rng = O.XorShiftRng()
    n, k0, d = 3000, 9, 4
    sc = rand_scalars(rng, cv.order, n)
    for table in (False, True):
        g_raw = G.Generators.progression(cid, k0, d, n, table=table, raw_jacobian=True)
        g_nrm = G.Generators.progression(cid, k0, d, n, table=table)
        raw, nrm = g_raw.commit_bytes(O.fes_to_bytes(sc, cv.order)), g_nrm.commit_bytes(O.fes_to_bytes(sc, cv.order))
        assert raw != nrm and O.jac_from_bytes(cv, raw) == O.jac_from_bytes(cv, nrm) == cv.msm_known_dlog(sc, k0, d)
        assert O.fe_from_bytes(nrm[64:96], cv.base) == 1
        assert g_raw.commit_bytes(O.fes_to_bytes([0] * 10, cv.order)) == bytes(96)


def test_msm_submit_wait(gpu_lib):
    """Asynchronous host-scalar MSM: two slots in flight give the same bytes as the synchronous call; slot misuse
    is reported."""
    import torch

    from vdf_b200 import VdfGpuError, _lib
    cv = O.PALLAS
    rng = O.XorShiftRng()
    n, k0, d = 20000, 11, 3
    g = G.Generators.progression(cv.cid, k0, d, n, table=True)
    vecs = [rand_scalars(rng, cv.order, n), rand_scalars(rng, cv.order, n - 7), rand_scalars(rng, cv.order, 100)]
    want = [g.commit_bytes(O.fes_to_bytes(v, cv.order)) for v in vecs]
    hosts = [torch.frombuffer(bytearray(O.fes_to_bytes(v, cv.order)), dtype=torch.uint8).pin_memory() for v in vecs]
    outs = [torch.zeros(96, dtype=torch.uint8).pin_memory() for _ in vecs]
    _lib.check(gpu_lib.vdfgpu_msm_submit(g._h, hosts[0].data_ptr(), len(vecs[0]), outs[0].data_ptr(), 0))
    _lib.check(gpu_lib.vdfgpu_msm_submit(g._h, hosts[1].data_ptr(), len(vecs[1]), outs[1].data_ptr(), 1))
    assert gpu_lib.vdfgpu_msm_submit(g._h, hosts[2].data_ptr(), len(vecs[2]), outs[2].data_ptr(), 1) == -3  # busy
    _lib.check(gpu_lib.vdfgpu_msm_wait(0))
    _lib.check(gpu_lib.vdfgpu_msm_submit(g._h, hosts[2].data_ptr(), len(vecs[2]), outs[2].data_ptr(), 0))
    _lib.check(gpu_lib.vdfgpu_msm_wait(1))
    _lib.check(gpu_lib.vdfgpu_msm_wait(0))
    assert [bytes(o.numpy().tobytes()) for o in outs] == want
    with pytest.raises(VdfGpuError):
        _lib.check(gpu_lib.vdfgpu_msm_wait(0))      # nothing in flight
    with pytest.raises(VdfGpuError):
        _lib.check(gpu_lib.vdfgpu_msm_submit(g._h, hosts[0].data_ptr(), n, outs[0].data_ptr(), 9))


@pytest.mark.gpu
@pytest.mark.parametrize("cid", CURVES)
@pytest.mark.parametrize("table", [False, True])
def test_msm_equal_points_special_cases_of_the_group_law(gpu_lib, cid, table):
    """Every generator the same point P: every bucket sum is a multiple of P, so the tree sums of the bucket reduction
    (quad additions, csrc/quad.cuh) keep meeting P + P (the doubling branch), and with P, -P alternating under equal
    scalars every bucket cancels to the identity (the identity branches).  Expected: (sum of the scalars) * P."""
    cv = O.CURVES[cid]
    n = 4096
    P = cv.mul(77, cv.gen)
    # distinct small scalars: bucket j of window 0 receives exactly one copy of P
    sc = [i + 1 for i in range(n)]
    g = G.Generators.from_points(cid, [P] * n, table=table)
    assert g.commit(sc) == cv.mul(sum(sc) % cv.order, P)
    # the same scalar everywhere: one bucket per window holds n * P, all others are empty
    s = (1 << 200) + 12345
    assert g.commit([s] * n) == cv.mul(s * n % cv.order, P)
    g.close()
    # P, -P, P, -P ... with pairwise equal scalars: everything cancels
    rng = O.XorShiftRng()
    half = rand_scalars(rng, cv.order, n // 2)
    sc2 = [half[i // 2] for i in range(n)]
    g = G.Generators.from_points(cid, [P if i % 2 == 0 else cv.neg(P) for i in range(n)], table=table)
    assert g.commit(sc2) is None
    # ... and with one survivor
    sc2[-1] = (sc2[-1] + 5) % cv.order
    assert g.commit(sc2) == cv.mul(cv.order - 5, P)
    g.close()
