"""GPU: the entry points on caller-owned streams and threads.

Every other GPU test synchronises the device around a call or goes through a host entry point that waits.  Here each
call runs on a stream the caller owns (vdfgpu_set_stream) behind a device delay of ~25 ms, far longer than the library
needs to enqueue, and nothing synchronises between the work that writes its inputs and the call.  Every device input
first holds *stale* contents: a valid input of the same shape whose answer differs.  On the caller stream s come the
delay, a device-to-device copy of the *fresh* contents and a sentinel fill of every device output, then the call with
s set, then the read-back on s.  A kernel or copy enqueued on any stream but s runs before the delay ends: it reads the
stale input or has its output overwritten by the sentinel, and the answer is wrong.

The resident running instance (vdfgpu_running) and the witness bank carry state from call to call: their cases switch
stream or thread between calls and check that each call sees the work of the previous one.
"""
import ctypes
import random
import threading

import pytest

from oracle import pasta as O
from tests import shape_gen as S
from tests.sat_ref import unsat_rows
from vdf_b200 import _lib
from vdf_b200 import msm as G
from vdf_b200 import nova as N
from vdf_b200 import spartan as SP

pytestmark = pytest.mark.gpu

DELAY_MS = 25
SENTINEL = 0xA5
K0, D = 555, 77
N_GRAPH = 13904        # a Nova-size commitment: replayed as a cached CUDA graph
N_BIG = 1 << 19        # above the graph-replay regime for every window size
_cycles_per_ms = []


def _calibrated():
    """Cycles of torch.cuda._sleep per millisecond, measured once with CUDA events."""
    import torch
    if not _cycles_per_ms:
        s = torch.cuda.Stream()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(s):
            torch.cuda._sleep(100_000)
            a.record()
            torch.cuda._sleep(20_000_000)
            b.record()
        b.synchronize()
        _cycles_per_ms.append(20_000_000 / a.elapsed_time(b))
    return _cycles_per_ms[0]


def delay(s, ms=DELAY_MS):
    """A kernel that spins for `ms` on stream s (it ends by itself)."""
    import torch
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(ms * _calibrated()))


@pytest.fixture
def lib(gpu_lib):
    """The library with the calling thread's stream reset to the library stream afterwards."""
    import torch
    _calibrated()
    try:
        yield gpu_lib
    finally:
        torch.cuda.synchronize()
        _lib.check(gpu_lib.vdfgpu_set_stream(None))


def set_stream(lib, s):
    _lib.check(lib.vdfgpu_set_stream(None if s is None else s.cuda_stream))


def dev(b):
    import torch
    return torch.frombuffer(bytearray(b or bytes(32)), dtype=torch.uint8).cuda()


def empty(nbytes):
    import torch
    return torch.full((nbytes,), SENTINEL ^ 0xFF, dtype=torch.uint8, device="cuda")


class Staged:
    """Device inputs that hold stale contents until stream s, behind a delay, copies the fresh ones in."""

    def __init__(self):
        self.pairs, self.outs = [], []

    def input(self, stale: bytes, fresh: bytes):
        assert len(stale) == len(fresh) and stale != fresh
        t = dev(stale)
        self.pairs.append((t, dev(fresh)))
        return t

    def output(self, nbytes):
        t = empty(nbytes)
        self.outs.append(t)
        return t

    def run(self, lib, s, fn, *args):
        """Call fn once on s and wait (a first launch can load modules and allocate workspaces, which may synchronise
        the device), then enqueue delay, fresh copies and sentinel fills on s and call fn with s set; no
        synchronisation between them."""
        import torch
        set_stream(lib, s)
        fn(*args)
        torch.cuda.synchronize()   # the stale contents are in place; from here on only s orders anything
        delay(s)
        with torch.cuda.stream(s):
            for dst, src in self.pairs:
                dst.copy_(src)
            for o in self.outs:
                o.fill_(SENTINEL)
        set_stream(lib, s)
        return fn(*args)


def readback(s, *tensors):
    """Copies on s, then s.synchronize()."""
    import torch
    with torch.cuda.stream(s):
        host = [t.to("cpu", non_blocking=True) for t in tensors]
    s.synchronize()
    return [h.numpy().tobytes() for h in host]


def fes(vals, m):
    return O.fes_to_bytes(vals, m)


def scalars(py, n, cv):
    return [py.randrange(cv.order) for _ in range(n)]


_GENS = {}


def gens_for(cid, table):
    if (cid, table) not in _GENS:
        _GENS[(cid, table)] = G.Generators.progression(cid, K0, D, N_BIG, table=table)
    return _GENS[(cid, table)]


def point(cv, b):
    return O.jac_from_bytes(cv, b)


# ---- a. every _dev entry point under a delayed caller stream --------------------------------------------------------
@pytest.mark.parametrize("table", [False, True])
@pytest.mark.parametrize("n", [N_GRAPH, N_BIG])
def test_msm_dev(lib, table, n):
    import torch
    cid = O.CURVE_PALLAS
    cv = O.CURVES[cid]
    g = gens_for(cid, table)
    py = random.Random(n + table)
    stale, fresh = scalars(py, n, cv), scalars(py, n, cv)
    st = Staged()
    sc = st.input(fes(stale, cv.order), fes(fresh, cv.order))
    out = st.output(96)
    s = torch.cuda.Stream()
    st.run(lib, s, lambda: _lib.check(lib.vdfgpu_msm_dev(g._h, sc.data_ptr(), n, out.data_ptr())))
    (got,) = readback(s, out)
    assert point(cv, got) == cv.msm_known_dlog(fresh, K0, D)


@pytest.mark.parametrize("lens", [(N_GRAPH, 9001), (N_GRAPH, 5, 12000, N_GRAPH)])
def test_msm_batch_dev(lib, lens):
    import torch
    cid = O.CURVE_VESTA
    cv = O.CURVES[cid]
    g = G.Generators.progression(cid, K0, D, N_GRAPH, table=True)
    py = random.Random(len(lens))
    st = Staged()
    fresh, ins = [], []
    for n in lens:
        a, b = scalars(py, n, cv), scalars(py, n, cv)
        ins.append(st.input(fes(a, cv.order), fes(b, cv.order)))
        fresh.append(b)
    out = st.output(96 * len(lens))
    k = len(lens)
    ptrs = (ctypes.c_void_p * k)(*[t.data_ptr() for t in ins])
    ln = (ctypes.c_size_t * k)(*lens)
    s = torch.cuda.Stream()
    st.run(lib, s, lambda: _lib.check(lib.vdfgpu_msm_batch_dev(g._h, ptrs, ln, k, out.data_ptr())))
    (got,) = readback(s, out)
    for j in range(k):
        assert point(cv, got[96 * j:96 * j + 96]) == cv.msm_known_dlog(fresh[j], K0, D), j
    g.close()


def test_msm_range_dev(lib):
    import torch
    cid = O.CURVE_PALLAS
    cv = O.CURVES[cid]
    g = gens_for(cid, False)
    first, n = 1234, N_GRAPH
    py = random.Random(first)
    stale, fresh = scalars(py, n, cv), scalars(py, n, cv)
    st = Staged()
    sc = st.input(fes(stale, cv.order), fes(fresh, cv.order))
    out = st.output(96)
    s = torch.cuda.Stream()
    st.run(lib, s, lambda: _lib.check(lib.vdfgpu_msm_range_dev(g._h, first, sc.data_ptr(), n, out.data_ptr())))
    (got,) = readback(s, out)
    assert point(cv, got) == cv.msm_known_dlog(fresh, K0 + first * D, D)


def test_point_sum_dev(lib):
    import torch
    cid = O.CURVE_VESTA
    cv = O.CURVES[cid]
    pts = cv.progression(3, 5, 40)
    old = cv.progression(4, 9, 40)
    want = None
    for p in pts:
        want = cv.add(want, p)
    st = Staged()
    inp = st.input(b"".join(O.jac_to_bytes(cv, p) for p in old), b"".join(O.jac_to_bytes(cv, p) for p in pts))
    out = st.output(96)
    s = torch.cuda.Stream()
    st.run(lib, s, lambda: _lib.check(lib.vdfgpu_point_sum_dev(cid, inp.data_ptr(), 40, out.data_ptr())))
    (got,) = readback(s, out)
    assert point(cv, got) == want


def _gpu_shape(fid, shape):
    return N.R1CSShape(fid, shape.num_cons, shape.num_vars, shape.num_io, shape.A, shape.B, shape.C)


@pytest.mark.parametrize("cons,vars_,io", [(1337, 900, 2), (2003, 1500, 7)])
def test_r1cs_dev_entry_points(lib, cons, vars_, io):
    """multiply_vec_dev, cross_term_dev, r1cs_bind_rows_dev and fold_dev on a general shape whose constraints read X."""
    import torch
    fid = O.FIELD_FQ
    shape = S.general_shape(fid, cons, vars_, io)
    m = shape.m
    gs = _gpu_shape(fid, shape)
    h = gs._h
    py = random.Random(cons)

    def inst():
        return S.random_vec(py, m, vars_), py.randrange(2, m), S.random_vec(py, m, io)
    (W1o, u1o, X1o), (W1, u1, X1) = inst(), inst()
    (W2o, _, X2o), (W2, _, X2) = inst(), inst()
    s = torch.cuda.Stream()

    st = Staged()
    Wd, uXd = st.input(fes(W1o, m), fes(W1, m)), st.input(fes([u1o] + X1o, m), fes([u1] + X1, m))
    abc = st.output(3 * cons * 32)
    st.run(lib, s, lambda: _lib.check(lib.vdfgpu_multiply_vec_dev(h, Wd.data_ptr(), uXd.data_ptr(), abc.data_ptr())))
    Az, Bz, Cz = shape.multiply_vec(shape.z_of(W1, u1, X1))
    assert O.fes_from_bytes(readback(s, abc)[0], m) == Az + Bz + Cz

    st = Staged()
    W1d, uX1d = st.input(fes(W1o, m), fes(W1, m)), st.input(fes([u1o] + X1o, m), fes([u1] + X1, m))
    W2d, uX2d = st.input(fes(W2o, m), fes(W2, m)), st.input(fes([1] + X2o, m), fes([1] + X2, m))
    Td = st.output(cons * 32)
    st.run(lib, s, lambda: _lib.check(lib.vdfgpu_cross_term_dev(h, W1d.data_ptr(), uX1d.data_ptr(), W2d.data_ptr(),
                                                                uX2d.data_ptr(), Td.data_ptr())))
    T = shape.cross_term(W1, u1, X1, W2, X2)
    assert O.fes_from_bytes(readback(s, Td)[0], m) == T

    st = Staged()
    eqo, eq = S.random_vec(py, m, cons), S.random_vec(py, m, cons)
    ro, r_abc = [py.randrange(m) for _ in range(3)], [py.randrange(m) for _ in range(3)]
    eqd, rd = st.input(fes(eqo, m), fes(eq, m)), st.input(fes(ro, m), fes(r_abc, m))
    scratch, Mt = st.output(3 * cons * 32), st.output((vars_ + 1 + io) * 32)
    st.run(lib, s, lambda: _lib.check(lib.vdfgpu_r1cs_bind_rows_dev(h, eqd.data_ptr(), rd.data_ptr(), scratch.data_ptr(),
                                                                    Mt.data_ptr())))
    assert O.fes_from_bytes(readback(s, Mt)[0], m) == shape.bind_rows(eq, r_abc)

    # fold_dev works in place: W1 and E1 are inputs and outputs
    st = Staged()
    E1o, E1 = S.random_vec(py, m, cons), S.random_vec(py, m, cons)
    r_old, r = py.randrange(1 << 128), py.randrange(1 << 128)
    W1d, W2d = st.input(fes(W1o, m), fes(W1, m)), st.input(fes(W2o, m), fes(W2, m))
    E1d, Td = st.input(fes(E1o, m), fes(E1, m)), st.input(fes(E1o[::-1], m), fes(T, m))
    rd = st.input(fes([r_old], m), fes([r], m))
    st.run(lib, s, lambda: _lib.check(lib.vdfgpu_fold_dev(fid, W1d.data_ptr(), W2d.data_ptr(), vars_, E1d.data_ptr(),
                                                          Td.data_ptr(), cons, rd.data_ptr())))
    gotW, gotE = readback(s, W1d, E1d)
    assert (O.fes_from_bytes(gotW, m), O.fes_from_bytes(gotE, m)) == (O.fold_vec(W1, W2, r, m), O.fold_vec(E1, T, r, m))
    gs.close()


def test_is_sat_relaxed_dev(lib):
    """The counters start as the sentinel; the call must produce the exact count and first row of the fresh instance."""
    import numpy as np
    import torch
    fid = O.FIELD_FP
    shape = S.general_shape(fid, 2003, 1500, 7)
    m, cons = shape.m, shape.num_cons
    gs = _gpu_shape(fid, shape)
    W, E, u, X = S.relaxed_instance(shape)
    Eo = list(E)
    Eo[5] = (Eo[5] + 1) % m                       # stale: one violated row, row 5
    Ef = list(E)
    for row in (700, 1999, cons - 1):             # fresh: three violated rows, the first 700
        Ef[row] = (Ef[row] + 3) % m
    Xo = list(X)
    st = Staged()
    Wd = st.input(fes(W[::-1], m), fes(W, m))
    Ed = st.input(fes(Eo, m), fes(Ef, m))
    uXd = st.input(fes([u] + Xo[::-1], m), fes([u] + X, m))
    counts = st.output(16)
    s = torch.cuda.Stream()
    st.run(lib, s, lambda: gs.is_sat_relaxed_dev(Wd, Ed, uXd, counts))
    got = np.frombuffer(readback(s, counts)[0], dtype=np.uint64).tolist()
    bad = unsat_rows(shape, W, Ef, u, X)
    assert bad == [700, 1999, cons - 1]
    assert got == [3, 700]
    gs.close()


def test_eq_evals_and_poly_evaluate_dev(lib):
    import torch
    fid = O.FIELD_FQ
    m = O.MODULUS[fid]
    ell = 12
    py = random.Random(12)
    r = [py.randrange(m) for _ in range(ell)]
    st = Staged()
    out = st.output(32 << ell)
    s = torch.cuda.Stream()
    rb = fes(r, m)
    st.run(lib, s, lambda: _lib.check(lib.vdfgpu_eq_evals_dev(fid, _lib.as_ptr(rb), ell, out.data_ptr())))
    assert O.fes_from_bytes(readback(s, out)[0], m) == O.eq_evals(r, m)

    old, poly = [py.randrange(m) for _ in range(1 << ell)], [py.randrange(m) for _ in range(1 << ell)]
    st = Staged()
    pd = st.input(fes(old, m), fes(poly, m))
    res = bytearray(32)
    st.run(lib, s, lambda: _lib.check(lib.vdfgpu_poly_evaluate_dev(fid, pd.data_ptr(), _lib.as_ptr(rb), ell,
                                                                   _lib.as_ptr(res))))
    s.synchronize()
    assert O.fe_from_bytes(bytes(res), m) == O.poly_evaluate(poly, r, m)


@pytest.mark.parametrize("ntab,ell", [(4, 10), (2, 11)])
def test_sumcheck_dev(lib, ntab, ell):
    """The tables are written late on s; every round's evaluations, as the callback receives them, match the oracle."""
    import torch
    fid = O.FIELD_FP
    m = O.MODULUS[fid]
    py = random.Random(ntab * 100 + ell)
    old = [[py.randrange(m) for _ in range(1 << ell)] for _ in range(ntab)]
    tabs = [[py.randrange(m) for _ in range(1 << ell)] for _ in range(ntab)]

    def challenge(rnd, evals):
        return (sum(evals) * 0x9E3779B97F4A7C15 + rnd + 777) % m
    want = O.sumcheck_prove(tabs, m, challenge)
    st = Staged()
    ins = [st.input(fes(a, m), fes(b, m)) for a, b in zip(old, tabs)]
    log = []
    cb = SP._round_trampoline(m, challenge, log)
    final = bytearray(32 * ntab)
    fn = lib.vdfgpu_sumcheck_cubic_dev if ntab == 4 else lib.vdfgpu_sumcheck_quad_dev
    s = torch.cuda.Stream()
    st.run(lib, s, lambda: _lib.check(fn(fid, *[t.data_ptr() for t in ins], ell, ctypes.cast(cb, ctypes.c_void_p), None,
                                         _lib.as_ptr(final))))
    s.synchronize()
    log = log[ell:]   # the rounds of the warm-up call on the stale tables come first
    assert [e for e, _ in log] == [tuple(e) for e in want[0]]
    assert [r for _, r in log] == want[1]
    assert O.fes_from_bytes(bytes(final), m) == want[2]


@pytest.mark.parametrize("fid,mk", [(O.FIELD_FQ, O.PallasVDF), (O.FIELD_FP, O.VestaVDF)])
def test_minroot_check_batch_dev(lib, fid, mk):
    """Per-chain t on the device and a uniform t; the stale originals give a different verdict vector."""
    import numpy as np
    import torch
    vdf = mk()
    m = vdf.m
    rng = O.XorShiftRng()
    n = 300
    res = [O.State(O.field_random(rng, m), O.field_random(rng, m), O.field_random(rng, m)) for _ in range(n)]
    ts = [[0, 1, 3, 8, 21][k % 5] for k in range(n)]
    ts_old = [[2, 0, 5, 1, 4][k % 5] for k in range(n)]

    def originals(t_of, bad):
        out = []
        for k, r in enumerate(res):
            o = vdf.inverse_eval(r, t_of(k))
            out.append(O.State((o.x + 1) % m, o.y, o.i) if bad(k) else o)
        return b"".join(O.state_to_bytes(o, m) for o in out)
    rb = b"".join(O.state_to_bytes(r, m) for r in res)
    rb_old = b"".join(O.state_to_bytes(O.State(r.y, r.x, r.i), m) for r in res)
    s = torch.cuda.Stream()
    st = Staged()
    rd = st.input(rb_old, rb)
    od = st.input(originals(lambda k: ts[k], lambda k: k % 5 == 1), originals(lambda k: ts[k], lambda k: k % 7 == 3))
    td = st.input(np.array(ts_old, np.uint64).tobytes(), np.array(ts, np.uint64).tobytes())
    ok = st.output(n)
    st.run(lib, s, lambda: _lib.check(lib.vdfgpu_minroot_check_batch_dev(fid, rd.data_ptr(), od.data_ptr(), td.data_ptr(),
                                                                         0, n, ok.data_ptr())))
    assert list(readback(s, ok)[0]) == [0 if k % 7 == 3 else 1 for k in range(n)]
    # one t for every chain
    st = Staged()
    rd = st.input(rb_old, rb)
    od = st.input(originals(lambda k: 8, lambda k: k % 4 == 0), originals(lambda k: 8, lambda k: k % 9 == 0))
    ok = st.output(n)
    st.run(lib, s, lambda: _lib.check(lib.vdfgpu_minroot_check_batch_dev(fid, rd.data_ptr(), od.data_ptr(), None, 8, n,
                                                                         ok.data_ptr())))
    assert list(readback(s, ok)[0]) == [0 if k % 9 == 0 else 1 for k in range(n)]


# ---- b. graph replay across streams ---------------------------------------------------------------------------------
def test_graph_replay_alternating_streams(lib):
    """One generator set, the same device scalar and output pointers, streams A, B, A, B with fresh data each time:
    a cached graph must be replayed on the stream of the call, not on the one it was captured on."""
    import torch
    cid = O.CURVE_PALLAS
    cv = O.CURVES[cid]
    g = gens_for(cid, True)
    A, B = torch.cuda.Stream(), torch.cuda.Stream()
    assert A.cuda_stream != B.cuda_stream
    py = random.Random(99)
    vecs = [scalars(py, N_GRAPH, cv) for _ in range(5)]
    sc = dev(fes(vecs[0], cv.order))
    out = empty(96)
    fresh = [dev(fes(v, cv.order)) for v in vecs[1:]]
    for k, s in enumerate((A, B, A, B)):
        st = Staged()
        st.pairs.append((sc, fresh[k]))
        st.outs.append(out)
        st.run(lib, s, lambda: _lib.check(lib.vdfgpu_msm_dev(g._h, sc.data_ptr(), N_GRAPH, out.data_ptr())))
        (got,) = readback(s, out)
        assert point(cv, got) == cv.msm_known_dlog(vecs[k + 1], K0, D), k


# ---- c. the headline configuration: back-to-back MSMs on several caller streams ------------------------------------
def _many_streams(lib, g, cv, sizes, rounds, seed):
    """Every (stream, round) gets its own scalars and output, behind a delay on that stream; no synchronisation until
    every call is enqueued."""
    import torch
    streams = [torch.cuda.Stream() for _ in sizes]
    assert len({s.cuda_stream for s in streams}) == len(streams)
    py = random.Random(seed)
    jobs = []
    for rnd in range(rounds):
        for s, n in zip(streams, sizes):
            v = scalars(py, n, cv)
            jobs.append((s, n, v, dev(fes(scalars(py, n, cv), cv.order)), dev(fes(v, cv.order)), empty(96)))
    torch.cuda.synchronize()
    for s, n, _, sc, fresh, out in jobs:
        delay(s, DELAY_MS / 5)
        with torch.cuda.stream(s):
            sc.copy_(fresh)
            out.fill_(SENTINEL)
        set_stream(lib, s)
        _lib.check(lib.vdfgpu_msm_dev(g._h, sc.data_ptr(), n, out.data_ptr()))
    for s, n, v, _, _, out in jobs:
        (got,) = readback(s, out)
        assert point(cv, got) == cv.msm_known_dlog(v, K0, D), n


def test_four_streams_back_to_back(lib):
    cid = O.CURVE_PALLAS
    _many_streams(lib, gens_for(cid, True), O.CURVES[cid], [1 << 16, 1 << 17, 3 << 16, 1 << 18], 1, 4)


def test_ten_streams_evict_workspaces(lib):
    """More streams than the 8 workspaces the library keeps: arenas are evicted while other streams have work in
    flight, and cached graphs of evicted arenas must not be replayed."""
    cid = O.CURVE_VESTA
    g = G.Generators.progression(cid, K0, D, N_GRAPH, table=True)
    _many_streams(lib, g, O.CURVES[cid], [N_GRAPH - k for k in range(10)], 2, 10)
    g.close()


# ---- d. host entry points on a busy caller stream --------------------------------------------------------------------
def test_host_entry_points_on_a_busy_stream(lib):
    """Each returns only after its own result has landed, although s still holds a pending delay."""
    import torch
    cid = O.CURVE_PALLAS
    cv = O.CURVES[cid]
    g = gens_for(cid, False)
    s = torch.cuda.Stream()
    set_stream(lib, s)
    py = random.Random(5)
    v = scalars(py, 20000, cv)
    delay(s)
    assert g.commit(v) == cv.msm_known_dlog(v, K0, D)
    pts = bytearray(b"".join(O.affine_to_bytes(cv, p) for p in cv.progression(K0, D, 3000)))
    _lib.check(lib.vdfgpu_dropin_cache_clear())
    for k, want_hit in enumerate((False, True)):
        w = scalars(py, 3000, cv)
        hits, misses, entries = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint64()
        _lib.check(lib.vdfgpu_dropin_cache_stats(ctypes.byref(hits), ctypes.byref(misses), ctypes.byref(entries)))
        h0, m0 = hits.value, misses.value
        delay(s)
        out = G.mult_pippenger(cid, pts, fes(w, cv.order))
        assert point(cv, out) == cv.msm_known_dlog(w, K0, D), k
        _lib.check(lib.vdfgpu_dropin_cache_stats(ctypes.byref(hits), ctypes.byref(misses), ctypes.byref(entries)))
        assert (hits.value - h0, misses.value - m0) == ((1, 0) if want_hit else (0, 1)), k
    fid = O.FIELD_FQ
    shape = S.general_shape(fid, 1337, 900, 2)
    gs = _gpu_shape(fid, shape)
    gsets = G.Generators.progression(cid, K0, D, 1337, table=True)
    W, E, u, X = S.relaxed_instance(shape)
    E[1000] = (E[1000] + 1) % shape.m
    U = N.RelaxedR1CSInstance(cv.msm_known_dlog(W, K0, D), cv.msm_known_dlog(E, K0, D), X, u)
    delay(s)
    rep = gs.is_sat_relaxed(gsets, W, E, U)
    assert (rep.bad_rows, rep.first_bad_row, rep.comm_W_ok, rep.comm_E_ok) == (1, 1000, True, True)
    gs.close()
    gsets.close()


# ---- e. resident handles across streams and threads -----------------------------------------------------------------
FID, CID = O.FIELD_FQ, O.CURVE_PALLAS


class Chain:
    """The IO-bound step instance (t = 5) and a device-resident running instance over it, with the oracle's fold."""

    def __init__(self, lib):
        self.lib = lib
        self.cv = O.CURVES[CID]
        self.steps = [S.fresh_instance(FID, 5, k, 64) for k in range(5)]
        self.shape = self.steps[0][0]
        self.m = self.shape.m
        self.gs = _gpu_shape(FID, self.shape)
        self.gens = G.Generators.progression(CID, K0, D, max(self.shape.num_cons, self.shape.num_vars), table=True)
        self.prover = N.RunningProver(self.gs, self.gens)
        _, W0, X0 = self.steps[0]
        self.Wr, self.Er, self.ur, self.Xr = list(W0), [0] * self.shape.num_cons, 1, list(X0)

    def set_running(self):
        self.prover.set_running(self.Wr, self.Er, N.RelaxedR1CSInstance(None, None, self.Xr, self.ur))

    def commit(self, k):
        """running_commit of step k (returns once comm_W2 and comm_T have landed); checks both commitments."""
        _, W2, X2 = self.steps[k]
        cW, cT = bytearray(96), bytearray(96)
        _lib.check(self.lib.vdfgpu_running_commit(self.prover._h, _lib.as_ptr(fes(W2, self.m)), _lib.as_ptr(fes(X2, self.m)),
                                                  _lib.as_ptr(cW), _lib.as_ptr(cT)))
        T = self.shape.cross_term(self.Wr, self.ur, self.Xr, W2, X2)
        assert point(self.cv, bytes(cW)) == self.cv.msm_known_dlog(W2, K0, D)
        assert point(self.cv, bytes(cT)) == self.cv.msm_known_dlog(T, K0, D), "comm_T"
        return T, point(self.cv, bytes(cT))

    def finish(self, k, T, r):
        _, W2, X2 = self.steps[k]
        _lib.check(self.lib.vdfgpu_running_finish(self.prover._h, _lib.as_ptr(fes([r], self.m))))
        m = self.m
        self.Wr, self.Er = O.fold_vec(self.Wr, W2, r, m), O.fold_vec(self.Er, T, r, m)
        self.ur, self.Xr = (self.ur + r) % m, O.fold_vec(self.Xr, X2, r, m)

    def want(self):
        return self.Wr, self.Er, self.ur, self.Xr

    def check_words(self):
        rep = (ctypes.c_uint64 * 4)()
        cW = O.jac_to_bytes(self.cv, self.cv.msm_known_dlog(self.Wr, K0, D))
        cE = O.jac_to_bytes(self.cv, self.cv.msm_known_dlog(self.Er, K0, D))
        _lib.check(self.lib.vdfgpu_running_check(self.prover._h, _lib.as_ptr(cW), _lib.as_ptr(cE), rep))
        return list(rep)

    def close(self):
        self.prover.close()
        self.gs.close()
        self.gens.close()


R1, R2 = 0x1F2E3D4C5B6A79880123456789ABCDEF, 0x0FEDCBA987654321F0E1D2C3B4A59687


@pytest.mark.parametrize("to", ["B", "library"])
@pytest.mark.parametrize("then", ["get", "check", "commit", "set"])
def test_running_after_a_stream_switch(lib, then, to):
    """With stream A set: set_running, running_commit, a delay on A, running_finish (which returns at once).  Then the
    next call on stream B or on the library stream must see the folded instance."""
    import torch
    c = Chain(lib)
    A, B = torch.cuda.Stream(), torch.cuda.Stream()
    target = B if to == "B" else None
    # a first check on the target stream, so that the checked one allocates no workspace (which may synchronise)
    set_stream(lib, target)
    c.set_running()
    c.prover.U = N.RelaxedR1CSInstance(c.cv.msm_known_dlog(c.Wr, K0, D), bytes(96), c.Xr, c.ur)
    rep = c.prover.check()
    assert [rep.bad_rows, rep.comm_W_ok, rep.comm_E_ok] == [0, True, True]
    set_stream(lib, A)
    c.set_running()
    comm_W0 = c.cv.msm_known_dlog(c.Wr, K0, D)
    T, comm_T = c.commit(1)
    comm_W = N.point_fold(CID, comm_W0, c.cv.msm_known_dlog(c.steps[1][1], K0, D), R1)
    comm_E = N.point_fold(CID, None, comm_T, R1)
    delay(A)
    c.finish(1, T, R1)
    set_stream(lib, target)
    if then == "get":
        assert c.prover.get_running() == c.want()
    elif then == "check":
        assert comm_W == c.cv.msm_known_dlog(c.Wr, K0, D) and comm_E == c.cv.msm_known_dlog(c.Er, K0, D)
        c.prover.U = N.RelaxedR1CSInstance(comm_W, comm_E, c.Xr, c.ur)
        rep = c.prover.check()
        assert [rep.bad_rows, rep.first_bad_row, rep.comm_W_ok, rep.comm_E_ok] == [0, None, True, True]
    elif then == "commit":
        T2, _ = c.commit(2)
        c.finish(2, T2, R2)
        assert c.prover.get_running() == c.want()
        assert unsat_rows(c.shape, *c.want()) == []
    else:
        py = random.Random(3)
        new = (S.random_vec(py, c.m, c.shape.num_vars), S.random_vec(py, c.m, c.shape.num_cons), 12345,
               S.random_vec(py, c.m, c.shape.num_io))
        c.prover.set_running(new[0], new[1], N.RelaxedR1CSInstance(None, None, new[3], new[2]))
        torch.cuda.synchronize()   # whatever was pending on A has run by now
        assert c.prover.get_running() == new
    c.close()


def test_running_prover_and_verifier_threads(lib):
    """A prover thread on stream A runs three fold steps, the last finish behind a delay; after join, a verifier
    thread on stream B checks the running instance in place."""
    import torch
    c = Chain(lib)
    A, B = torch.cuda.Stream(), torch.cuda.Stream()
    errors, report = [], []

    def prover():
        try:
            set_stream(lib, A)
            c.set_running()
            for k in (1, 2, 3):
                T, _ = c.commit(k)
                if k == 3:
                    delay(A)
                c.finish(k, T, R1 + k)
        except Exception as e:   # surfaces in the main thread
            errors.append(e)

    def verifier():
        try:
            set_stream(lib, B)
            report.append(c.check_words())
            _lib.check(lib.vdfgpu_set_stream(None))
        except Exception as e:
            errors.append(e)
    for fn in (prover, verifier):
        th = threading.Thread(target=fn)
        th.start()
        th.join()
    assert not errors, errors
    assert report == [[0, c.shape.num_cons, 1, 1]]
    assert unsat_rows(c.shape, *c.want()) == []
    c.close()


def test_is_sat_relaxed_from_three_threads(lib):
    """Three threads, each with its own stream, check the same two shape handles at once; one instance has a corrupted
    E entry.  Each report must be exact."""
    import torch
    cv = O.CURVES[CID]
    shapes = [S.general_shape(FID, 1337, 900, 2), S.general_shape(FID, 2003, 1500, 7)]
    gss = [_gpu_shape(FID, sh) for sh in shapes]
    gens = G.Generators.progression(CID, K0, D, 2003, table=True)
    cases = []
    for j, sh in enumerate(shapes):
        W, E, u, X = S.relaxed_instance(sh, seed=j + 7)
        if j == 1:
            E[1500] = (E[1500] + 1) % sh.m
        U = N.RelaxedR1CSInstance(cv.msm_known_dlog(W, K0, D), cv.msm_known_dlog(E, K0, D), X, u)
        cases.append((W, E, U, (1, 1500) if j else (0, None)))
    start = threading.Barrier(3)
    errors, reports = [], {}

    def verify(tid):
        try:
            s = torch.cuda.Stream()
            set_stream(lib, s)
            start.wait()
            for rnd in range(3):
                for j in (0, 1):
                    delay(s, DELAY_MS / 5)
                    W, E, U, _ = cases[j]
                    rep = gss[j].is_sat_relaxed(gens, W, E, U)
                    reports[(tid, rnd, j)] = (rep.bad_rows, rep.first_bad_row, rep.comm_W_ok, rep.comm_E_ok)
            _lib.check(lib.vdfgpu_set_stream(None))
        except Exception as e:
            errors.append(e)
    threads = [threading.Thread(target=verify, args=(t,)) for t in range(3)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors
    assert len(reports) == 18
    for (tid, rnd, j), rep in reports.items():
        assert rep == cases[j][3] + (True, True), (tid, rnd, j)
    for g in gss:
        g.close()
    gens.close()


def test_witness_bank_consumed_at_once_from_other_streams(lib):
    """A bank at t = 16 384 takes milliseconds to generate.  running_commit_step is called right after the bank is
    created, from another stream, without a bank.read() first; witness_bank_read of a second bank right after its
    creation, from a third stream.  Both must see the generated witness."""
    import torch
    fid, cid = FID, CID
    cv = O.CURVES[cid]
    t = 16384
    per = 4 * t + 1
    rng = O.XorShiftRng(O.TEST_SEED)
    insts = [O.make_step_instance(fid, t, O.State(O.field_random(rng, O.MODULUS[fid]), 0, k + 1)) for k in range(3)]
    shape = insts[0][0]
    m = shape.m
    off = shape.num_vars - per
    states = [tuple(W[off - 3:off]) for _, W, _, _ in insts]
    gs = _gpu_shape(fid, shape)
    gens = G.Generators.progression(cid, K0, D, max(shape.num_cons, shape.num_vars), table=True)
    host, bankfed = N.RunningProver(gs, gens), N.RunningProver(gs, gens)
    U = N.RelaxedR1CSInstance(None, None, list(insts[0][2]), 1)
    for p in (host, bankfed):
        p.set_running(insts[0][1], [0] * shape.num_cons, U)
    _, W2, X2, _ = insts[2]
    full = O.fes_to_bytes(W2, m)
    holed = bytearray(full)
    holed[32 * off:32 * (off + per)] = b"\xee" * (32 * per)
    r = 0xFEDCBA9876543210
    a = host.prove_step_bytes(full, fes(X2, m), r)
    B, C = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    bank = N.WitnessBank(fid, states, t)
    set_stream(lib, B)
    b = bankfed.prove_step_bank_bytes(bank, 2, off, bytes(holed), fes(X2, m), r)
    assert O.jac_from_bytes(cv, b[0]) == cv.msm_known_dlog(W2, K0, D)
    assert a == b
    assert bankfed.get_running() == host.get_running()
    bank2 = N.WitnessBank(fid, states, t)
    set_stream(lib, C)
    assert bank2.read(1, 2) == [W[off:off + per] for _, W, _, _ in insts[1:]]
    for x in (host, bankfed, bank, bank2, gs, gens):
        x.close()
