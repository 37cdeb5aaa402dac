"""GPU: device-pointer entry points of the MSM and MinRoot paths that no other test calls -- vdfgpu_msm_dev,
vdfgpu_msm_range_dev (the per-rank MSM of the multi-GPU path), vdfgpu_point_sum_dev and
vdfgpu_minroot_check_batch_dev -- against the known-discrete-log identity and their host forms."""
import random

import pytest

from oracle import pasta as O
from tests.shape_gen import random_vec
from vdf_b200 import VdfGpuError, _lib
from vdf_b200 import msm as G

pytestmark = pytest.mark.gpu


def _to_dev(b):
    import torch
    return torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()


def _run(lib, fn, *args):
    import torch
    torch.cuda.synchronize()
    _lib.check(fn(*args))
    _lib.check(lib.vdfgpu_synchronize())


@pytest.mark.parametrize("cid", [O.CURVE_PALLAS, O.CURVE_VESTA])
@pytest.mark.parametrize("table", [False, True])
def test_msm_dev_and_range_dev(gpu_lib, cid, table):
    """P_i = (k0 + i d) G, so the range [first, first + n) commits to (sum_i s_i (k0 + (first + i) d)) G."""
    import torch
    lib = gpu_lib
    cv = O.CURVES[cid]
    k0, d, N = 555, 77, 6000
    py = random.Random(cid * 2 + table)
    g = G.Generators.progression(cid, k0, d, N, table=table)
    out = torch.zeros(96, dtype=torch.uint8, device="cuda")
    sc = random_vec(py, cv.order, 4099)
    scd = _to_dev(O.fes_to_bytes(sc, cv.order))
    for n in (4099, 1):
        _run(lib, lib.vdfgpu_msm_dev, g._h, scd.data_ptr(), n, out.data_ptr())
        assert O.jac_from_bytes(cv, out.cpu().numpy().tobytes()) == cv.msm_known_dlog(sc[:n], k0, d), n
    ranges = ((0, 4099), (1, 4099), (N - 4099, 4099), (1234, 777))
    for first, n in ranges:
        if table and first:
            with pytest.raises(VdfGpuError):   # a table set is sharded by creating one set per rank
                g.msm_dev(scd.data_ptr(), n, out.data_ptr(), first=first)
            continue
        _run(lib, lib.vdfgpu_msm_range_dev, g._h, first, scd.data_ptr(), n, out.data_ptr())
        assert O.jac_from_bytes(cv, out.cpu().numpy().tobytes()) == cv.msm_known_dlog(sc[:n], k0 + first * d, d), first
    if not table:   # past the end of the set
        with pytest.raises(VdfGpuError):
            g.msm_dev(scd.data_ptr(), 4099, out.data_ptr(), first=N - 4098)
    g.close()


@pytest.mark.parametrize("cid", [O.CURVE_PALLAS, O.CURVE_VESTA])
def test_point_sum_dev(gpu_lib, cid):
    import torch
    lib = gpu_lib
    cv = O.CURVES[cid]
    py = random.Random(11 + cid)
    pts = cv.progression(3, 5, 40)
    pts[7], pts[20] = None, cv.neg(pts[19])   # the identity; P + (-P)
    pts[30] = pts[29]                          # a doubling
    raw = []
    for p in pts:   # un-normalised Jacobian inputs (Z != 1) next to canonical ones
        if p is not None and py.random() < 0.5:
            z = py.randrange(2, cv.base)
            raw.append(O.fe_to_bytes(p[0] * z * z, cv.base) + O.fe_to_bytes(p[1] * z ** 3, cv.base) + O.fe_to_bytes(z, cv.base))
        else:
            raw.append(O.jac_to_bytes(cv, p))
    want = None
    for p in pts:
        want = cv.add(want, p)
    out = torch.zeros(96, dtype=torch.uint8, device="cuda")
    for k in (40, 33, 1, 0):
        _run(lib, lib.vdfgpu_point_sum_dev, cid, _to_dev(b"".join(raw[:k]) or bytes(96)).data_ptr(), k, out.data_ptr())
        host = G.point_sum(cid, b"".join(raw[:k]))
        w = None
        for p in pts[:k]:
            w = cv.add(w, p)
        assert O.jac_from_bytes(cv, out.cpu().numpy().tobytes()) == O.jac_from_bytes(cv, host) == w, k
    assert w is None and want is not None


@pytest.mark.parametrize("fid,mk", [(O.FIELD_FQ, O.PallasVDF), (O.FIELD_FP, O.VestaVDF)])
def test_minroot_check_batch_dev(gpu_lib, fid, mk):
    """Per-chain t (t_each on the device) and a uniform t; corrupted x, y or i in some originals."""
    import numpy as np
    import torch
    lib = gpu_lib
    vdf = mk()
    m = vdf.m
    rng = O.XorShiftRng()
    n = 300
    res, orig, ts = [], [], []
    for k in range(n):
        r = O.State(O.field_random(rng, m), O.field_random(rng, m), O.field_random(rng, m))
        t = [0, 1, 3, 8, 21][k % 5]
        o = vdf.inverse_eval(r, t)
        if k % 7 == 3:
            o = [O.State((o.x + 1) % m, o.y, o.i), O.State(o.x, (o.y + 1) % m, o.i), O.State(o.x, o.y, (o.i + 1) % m)][k % 3]
        res.append(r), orig.append(o), ts.append(t)
    rb = b"".join(O.state_to_bytes(s, m) for s in res)
    ob = b"".join(O.state_to_bytes(s, m) for s in orig)
    tb = np.array(ts, dtype=np.uint64)
    rd, od, td = _to_dev(rb), _to_dev(ob), _to_dev(tb.tobytes())
    ok = torch.full((n,), 7, dtype=torch.uint8, device="cuda")
    _run(lib, lib.vdfgpu_minroot_check_batch_dev, fid, rd.data_ptr(), od.data_ptr(), td.data_ptr(), 0, n, ok.data_ptr())
    want = [vdf.check(r, t, o) for r, t, o in zip(res, ts, orig)]
    assert [bool(v) for v in ok.cpu().tolist()] == want and want.count(False) == len(range(3, n, 7))
    host = np.zeros(n, np.uint8)
    _lib.check(lib.vdfgpu_minroot_check_batch(fid, _lib.as_ptr(rb), _lib.as_ptr(ob), tb.ctypes.data, 0, n, host.ctypes.data))
    assert host.tolist() == ok.cpu().tolist()
    # one t for every chain
    ob8 = b"".join(O.state_to_bytes(vdf.inverse_eval(r, 8) if k % 9 else O.State(0, 0, 0), m) for k, r in enumerate(res))
    _run(lib, lib.vdfgpu_minroot_check_batch_dev, fid, rd.data_ptr(), _to_dev(ob8).data_ptr(), None, 8, n, ok.data_ptr())
    assert [bool(v) for v in ok.cpu().tolist()] == [k % 9 != 0 for k in range(n)]
