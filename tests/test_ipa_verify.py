"""CPU: batch verification of inner-product arguments.  The scalar-table functors (sumcheck.cuh IpaHalfTablesFn,
IpaBatchScalarsFn) run by a CPU loop (tests/emul/emul_ipa_verify.cpp) against Python integers; spartan.ipa_b_hat's
closed form against <b, s>; the reference batch verifier (tests/ipa_verify_ref.py) against ipa_ref.verify; and the
argument errors of vdfgpu_ipa_verify_batch, which come back before any device work, with or without a GPU."""
import ctypes
import random
import subprocess
from pathlib import Path

import pytest

from oracle import pasta as O
from tests import ipa_ref as IR
from tests import ipa_verify_ref as VR
from tests.util import aligned, ptr
from vdf_b200 import _lib
from vdf_b200 import spartan as SP

ROOT = Path(__file__).resolve().parent.parent
SZ = ctypes.c_size_t
U32 = ctypes.c_uint32
ERR_ARG = -1


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    src = ROOT / "tests" / "emul" / "emul_ipa_verify.cpp"
    lib = tmp_path_factory.mktemp("emul_ipa_verify") / "libvdf_emul_ipa_verify.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", str(lib), str(src)],
                   check=True)
    return ctypes.CDLL(str(lib))


def _buf(vals, m):
    return aligned(O.fes_to_bytes(vals, m) or bytes(32))


def _vals(arr, count, m):
    return O.fes_from_bytes(arr.tobytes()[:32 * count], m)


# ---- the scalar table of the MSM over the resident set -------------------------------------------------------
@pytest.mark.parametrize("fid", [O.FIELD_FP, O.FIELD_FQ])
@pytest.mark.parametrize("ell", [0, 1, 2, 3, 7, 8])
@pytest.mark.parametrize("k", [1, 3, 5])
def test_scalar_table_matches_reference(emul, fid, ell, k):
    """S = sum_q w_q a_hat_q s_q and S[n] = the caller's value, through the Hi / Lo split (odd and even ell, empty
    halves at ell = 0 and ell = 1); challenges 1 and order - 1 among the random ones."""
    m = O.MODULUS[fid]
    py = random.Random(1000 * ell + 10 * k + fid)
    n = 1 << ell
    rs = [[py.randrange(1, m) for _ in range(ell)] for _ in range(k)]
    if ell:
        rs[0][0] = 1
        rs[-1][-1] = m - 1
    scales = [py.randrange(1, m) * py.randrange(1, m) % m for _ in range(k)]
    last = py.randrange(m)
    lo_bits = ell // 2
    hi_bits = ell - lo_bits
    r_b = _buf([r for row in rs for r in row], m)
    ri_b = _buf([pow(r, -1, m) for row in rs for r in row], m)
    hi, lo = aligned(bytes(32 * k << hi_bits)), aligned(bytes(32 * k << lo_bits))
    emul.emul_ipa_half_tables(fid, ptr(r_b), ptr(ri_b), ptr(_buf(scales, m)), U32(ell), U32(lo_bits), SZ(k), ptr(hi),
                              ptr(lo))
    got_hi, got_lo = _vals(hi, k << hi_bits, m), _vals(lo, k << lo_bits, m)
    for q in range(k):
        want_hi, want_lo = VR.half_tables(rs[q], scales[q], lo_bits, m)
        assert got_hi[q << hi_bits:(q + 1) << hi_bits] == want_hi, q
        assert got_lo[q << lo_bits:(q + 1) << lo_bits] == want_lo, q
    S = aligned(bytes(32 * (n + 1)))
    emul.emul_ipa_batch_scalars(fid, ptr(hi), ptr(lo), U32(hi_bits), U32(lo_bits), SZ(k), ptr(_buf([last], m)), ptr(S))
    got = _vals(S, n + 1, m)
    assert got[:n] == VR.batch_scalars(rs, scales, m)
    assert got[n] == last
    # one proof alone from the same tables (the single-proof checks of a failing batch)
    q = k - 1
    emul.emul_ipa_batch_scalars(fid, ptr(hi[32 * (q << hi_bits):]), ptr(lo[32 * (q << lo_bits):]), U32(hi_bits),
                                U32(lo_bits), SZ(1), ptr(_buf([last], m)), ptr(S))
    assert _vals(S, n, m) == [scales[q] * v % m for v in IR.s_table(rs[q], m)]


# ---- b_hat in closed form ------------------------------------------------------------------------------------
def _eq(x, m):
    ell = len(x)
    out = []
    for i in range(1 << ell):
        v = 1
        for j in range(ell):
            v = v * (x[j] if (i >> (ell - 1 - j)) & 1 else 1 - x[j]) % m
        out.append(v)
    return out


@pytest.mark.parametrize("fid", [O.FIELD_FP, O.FIELD_FQ])
def test_b_hat_closed_form(fid):
    m = O.MODULUS[fid]
    py = random.Random(7 + fid)
    ell = 6
    rs = [py.randrange(1, m) for _ in range(ell)]
    s = IR.s_table(rs, m)
    x1, x2 = [py.randrange(m) for _ in range(ell)], [py.randrange(m) for _ in range(ell)]
    rho = py.randrange(m)
    # one eq table
    assert SP.ipa_b_hat(fid, rs, [(1, x1)]) == IR.inner(_eq(x1, m), s, m)
    # two evaluation claims folded into one instance: b = eq(x1) + rho eq(x2)
    b = [(u + rho * v) % m for u, v in zip(_eq(x1, m), _eq(x2, m))]
    assert SP.ipa_b_hat(fid, rs, [(1, x1), (rho, x2)]) == IR.inner(b, s, m)
    # a shorter table zero-padded at the top, folded with a full one
    x3 = [py.randrange(m) for _ in range(ell - 2)]
    padded = _eq(x3, m) + [0] * (len(s) - (1 << len(x3)))
    assert SP.ipa_b_hat(fid, rs, [(rho, x3)]) == rho * IR.inner(padded, s, m) % m
    b = [(u + rho * v) % m for u, v in zip(_eq(x1, m), padded)]
    assert SP.ipa_b_hat(fid, rs, [(1, x1), (rho, x3)]) == IR.inner(b, s, m)
    # boolean points pick one entry of s
    assert SP.ipa_b_hat(fid, rs, [(1, [0, 1, 1, 0, 0, 1])]) == s[0b011001]
    assert SP.ipa_b_hat(fid, [], [(rho, [])]) == rho


# ---- the reference batch verifier against ipa_ref.verify -----------------------------------------------------
def _proofs(cv, G, U0, ell, k, seed):
    m = cv.order
    py = random.Random(seed)
    n = 1 << ell
    out = []
    for q in range(k):
        a = [py.randrange(m) for _ in range(n)]
        b = [py.randrange(m) for _ in range(n)]
        u_scale = py.randrange(1, m)
        salt = py.randrange(1 << 30)
        Ls, Rs, rs, a_hat = IR.prove(cv, G, U0, u_scale, a, b, lambda rnd, L, R, salt=salt: hash((salt, rnd, L, R)))
        b_hat = IR.inner(b, IR.s_table(rs, m), m)
        out.append(((Ls, Rs, rs, a_hat, cv.msm_naive(a, G), IR.inner(a, b, m), b_hat, u_scale), b))
    return out


def _ref_verify(cv, G, U0, proof, b):
    Ls, Rs, rs, a_hat, comm_a, c, _, u_scale = proof
    P = cv.add(comm_a, cv.mul(c * u_scale, U0))
    return IR.verify(cv, G, U0, u_scale, P, b, Ls, Rs, rs, a_hat)


@pytest.mark.parametrize("cid", [O.CURVE_PALLAS, O.CURVE_VESTA])
def test_reference_batch_verifier_agrees_with_ipa_ref(cid):
    cv = O.CURVES[cid]
    m = cv.order
    ell = 2
    py = random.Random(40 + cid)
    pts = [cv.mul(py.randrange(1, m), cv.gen) for _ in range((1 << ell) + 1)]
    G, U0 = pts[:-1], pts[-1]
    proofs = _proofs(cv, G, U0, ell, 3, 50 + cid)
    for p, b in proofs:
        assert VR.verify_one(cv, G, U0, p) and _ref_verify(cv, G, U0, p, b)
    good = [p for p, _ in proofs]
    w = [py.randrange(1, m) for _ in good]
    assert VR.batch_passes(cv, G, U0, good, w)
    # one corrupted field at a time: both verifiers reject that proof, the batch fails
    p, b = proofs[1]
    Ls, Rs, rs, a_hat, comm_a, c, b_hat, u_scale = p
    bad = [
        (Ls, Rs, rs, (a_hat + 1) % m, comm_a, c, b_hat, u_scale),
        ([cv.add(Ls[0], cv.gen)] + Ls[1:], Rs, rs, a_hat, comm_a, c, b_hat, u_scale),
        (Rs, Ls, rs, a_hat, comm_a, c, b_hat, u_scale),
        (Ls, Rs, rs, a_hat, cv.add(comm_a, cv.gen), c, b_hat, u_scale),
        (Ls, Rs, rs, a_hat, comm_a, (c + 1) % m, b_hat, u_scale),
        (Ls, Rs, rs, a_hat, comm_a, c, b_hat, (u_scale + 1) % m),
        (Ls, Rs, [rs[0] + 1] + rs[1:], a_hat, comm_a, c, b_hat, u_scale),
    ]
    for x in bad:
        assert not VR.verify_one(cv, G, U0, x) and not _ref_verify(cv, G, U0, x, b)
        assert not VR.batch_passes(cv, G, U0, [good[0], x, good[2]], w)
    # b_hat is checked only through the equation (ipa_ref.verify derives it from b)
    assert not VR.verify_one(cv, G, U0, (Ls, Rs, rs, a_hat, comm_a, c, (b_hat + 1) % m, u_scale))
    # two corruptions that cancel under equal weights: why the weights must be random
    d = cv.mul(py.randrange(1, m), cv.gen)
    p0, p2 = list(good[0]), list(good[2])
    p0[4], p2[4] = cv.add(p0[4], d), cv.add(p2[4], cv.neg(d))
    assert not VR.verify_one(cv, G, U0, p0) and not VR.verify_one(cv, G, U0, p2)
    assert VR.batch_passes(cv, G, U0, [p0, p2], [1, 1])
    assert not VR.batch_passes(cv, G, U0, [p0, p2], [w[0], w[2]])


# ---- argument errors: before any device work ------------------------------------------------------------------
class _FakeGens(ctypes.Structure):
    """The leading fields of struct vdfgpu_gens (vdf_b200/csrc/ctx.cuh): the argument checks read curve and n only,
    so a host-memory handle with many points reaches the challenge and weight checks without a GPU."""
    _fields_ = [("curve", ctypes.c_int), ("n", ctypes.c_size_t), ("flags", ctypes.c_uint32), ("c", ctypes.c_uint32),
                ("W", ctypes.c_uint32), ("pts", ctypes.c_void_p), ("refs", ctypes.c_int)]


_big = _FakeGens(O.CURVE_PALLAS, 1 << 20, 0, 0, 1, None, 0)
_empty = ctypes.create_string_buffer(1 << 12)   # zeroed: a set of 0 points
M = O.Q   # Pallas scalars
ELL, K = 2, 2
_pts = O.jac_to_bytes(O.PALLAS, O.PALLAS.gen) * (K * ELL)
_one = O.fes_to_bytes([1] * (K * ELL), M)


def _args(**over):
    a = dict(g=ctypes.addressof(_big), ell=ELL, k=K, comm=_pts, L=_pts, R=_pts, r=_one, a_hat=_one, c=_one,
             b_hat=_one, u_scale=_one, w=_one, ok=bytearray(K))
    a.update(over)
    return a


def _call(lib, a):
    p = _lib.as_ptr
    return lib.vdfgpu_ipa_verify_batch(a["g"], a["ell"], a["k"], p(a["comm"]), p(a["L"]), p(a["R"]), p(a["r"]),
                                       p(a["a_hat"]), p(a["c"]), p(a["b_hat"]), p(a["u_scale"]), p(a["w"]),
                                       p(a["ok"]))


def _with(raw32: bytes, at: int):
    """_one with element `at` replaced by 32 raw bytes"""
    return _one[:32 * at] + raw32 + _one[32 * (at + 1):]


_CASES = {
    "null gens": _args(g=None),
    "null comm_a": _args(comm=None),
    "null L": _args(L=None),
    "null R": _args(R=None),
    "null r": _args(r=None),
    "null a_hat": _args(a_hat=None),
    "null c": _args(c=None),
    "null b_hat": _args(b_hat=None),
    "null u_scale": _args(u_scale=None),
    "null w": _args(w=None),
    "null ok": _args(ok=None),
    "k = 0": _args(k=0),
    "ell 41": _args(ell=41),
    "too few points": _args(g=ctypes.addressof(_empty)),
    "challenge 0": _args(r=_with(bytes(32), 3)),
    "challenge = order": _args(r=_with(M.to_bytes(32, "little"), 1)),
    "challenge > order": _args(r=_with((M + 1).to_bytes(32, "little"), 0)),
    "weight 0": _args(w=_with(bytes(32), 1)),
    "weight = order": _args(w=_with(M.to_bytes(32, "little"), 0)),
    "weight all ones": _args(w=_with(b"\xff" * 32, 0)),
}


@pytest.mark.parametrize("case", sorted(_CASES))
def test_argument_errors_launch_nothing(case):
    lib = _lib.load()
    launches = lib.vdfgpu_launch_count()
    assert _call(lib, _CASES[case]) == ERR_ARG, lib.vdfgpu_last_error()
    assert lib.vdfgpu_last_error().decode().startswith("ipa_verify_batch: ")
    assert lib.vdfgpu_launch_count() == launches


def test_malformed_proofs_are_verdicts_not_errors():
    """Every proof malformed: the call succeeds with verdicts 0 and no device work -- off-curve points, coordinates
    >= p, a non-canonical a_hat -- while NULL L, R and r are fine at ell = 0."""
    lib = _lib.load()
    launches = lib.vdfgpu_launch_count()
    cv = O.PALLAS
    g = cv.mul(5, cv.gen)
    good = O.jac_to_bytes(cv, g)
    off_curve = good[:32] + O.fe_to_bytes(g[1] + 1, cv.base) + good[64:]
    big_x = O.P.to_bytes(32, "little") + good[32:]
    big_z = good[:64] + (O.P + 1).to_bytes(32, "little")
    comm = off_curve + big_x + big_z + good
    k = 4
    ones = O.fes_to_bytes([1] * k, M)
    a_hat = ones[:96] + M.to_bytes(32, "little")
    ok = bytearray(b"\x07" * k)
    p = _lib.as_ptr
    rc = lib.vdfgpu_ipa_verify_batch(ctypes.addressof(_big), 0, k, p(comm), None, None, None, p(a_hat), p(ones),
                                     p(ones), p(ones), p(ones), p(ok))
    assert rc == 0, lib.vdfgpu_last_error()
    assert ok == bytes(k)
    assert lib.vdfgpu_launch_count() == launches


def test_verdicts_fail_closed_when_the_call_fails():
    """Three well-formed proofs pass the host checks, then the call fails for want of a device (VDFGPU_ERR_CUDA): no
    verdict may read 1 for proofs that were never checked.  Runs where no CUDA device is usable; on a GPU machine the
    host-memory handle would reach the device work, so the test is skipped there."""
    lib = _lib.load()
    if lib.vdfgpu_device_count() > 0:
        pytest.skip("a CUDA device is usable: the call would not fail")
    k = 3
    a = _args(k=k, ok=bytearray(b"\x07" * k), comm=_pts[:96 * k], L=_pts + _pts, R=_pts + _pts,
              r=O.fes_to_bytes([1] * (k * ELL), M), a_hat=_one[:32 * k], c=_one[:32 * k], b_hat=_one[:32 * k],
              u_scale=_one[:32 * k], w=_one[:32 * k])
    assert _call(lib, a) == -2, lib.vdfgpu_last_error()
    assert a["ok"] == bytes(k)


def test_python_mirror_rejects_points_that_are_not_96_bytes():
    """A 72-byte affine record or a short point would make the C side read past the joined buffer"""
    from types import SimpleNamespace
    gens = SimpleNamespace(curve=O.CURVE_PALLAS, _h=None)
    good = O.jac_to_bytes(O.PALLAS, O.PALLAS.gen)
    for comm, L in ((good[:72], good), (good, good[:64])):
        with pytest.raises(ValueError):
            SP.ipa_verify_batch(gens, [([L], [good], [1], 1, comm, 1, 1, 1)], weights=[1])
