"""GPU: Spartan of a resident running instance in one call (vdfgpu_running_spartan_prove) and the verifier's sparse
evaluation (vdfgpu_r1cs_evaluate), both fields/curves, against tests/spartan_ref.py: everything the callbacks receive
and a_hat byte for byte; acceptance by the sum-check verifier, vdfgpu_r1cs_evaluate and vdfgpu_ipa_verify_batch;
padded shapes; rejection; the instance left as it was; ordering across streams; two threads; callback failures and
handles destroyed during a call; Nova sizes."""
import random
import threading

import pytest

from oracle import pasta as O
from tests import shape_gen as S
from tests import spartan_ref as SR
from vdf_b200 import VdfGpuError, _lib
from vdf_b200 import msm as G
from vdf_b200 import nova as N
from vdf_b200 import spartan as SP

pytestmark = pytest.mark.gpu

K0, D = 1234567, 89
R_FOLD = 0x1F2E3D4C5B6A79880123456789ABCDEF
CURVE_OF = {O.FIELD_FQ: O.CURVE_PALLAS, O.FIELD_FP: O.CURVE_VESTA}   # the curve whose scalar field is the shape's
FIDS = [O.FIELD_FQ, O.FIELD_FP]


class Instance:
    """A shape on the device, a known-dlog set of m + 1 points (commitment generators and the IPA set at once) and a
    running prover holding (W, E, u, X); the same on the host (oracle), with comm_W and comm_E by known discrete logs."""

    def __init__(self, fid, shape, W, E, u, X):
        self.fid, self.shape, self.p = fid, shape, shape.m
        self.cid = CURVE_OF[fid]
        self.cv = O.CURVES[self.cid]
        self.m = SR.padded_size(shape)
        self.gens = G.Generators.progression(self.cid, K0, D, self.m + 1)
        self.gs = N.R1CSShape(fid, shape.num_cons, shape.num_vars, shape.num_io, shape.A, shape.B, shape.C)
        self.rp = N.RunningProver(self.gs, self.gens)
        self.set(W, E, u, X)
        self.tau = [random.Random(self.m).randrange(self.p) for _ in range(self.m.bit_length() - 1)]

    def set(self, W, E, u, X):
        self.W, self.E, self.u, self.X = list(W), list(E), u, list(X)
        self.rp.set_running(W, E, N.RelaxedR1CSInstance(None, None, list(X), u))

    @classmethod
    def folded_step(cls, fid, t, aug):
        """two step instances folded on the device: u = 1 + r, E = r T != 0"""
        shape, W1, X1, _ = O.make_step_instance(fid, t, O.State(5, 6, t), aug_cons=aug)
        _, W2, X2, _ = O.make_step_instance(fid, t, O.State(9, 1, t), aug_cons=aug)
        inst = cls(fid, shape, W1, [0] * shape.num_cons, 1, X1)
        inst.fold(W2, X2, R_FOLD)
        return inst

    def fold(self, W2, X2, r):
        p = self.p
        T = self.shape.cross_term(self.W, self.u, self.X, W2, X2)
        self.rp.prove_step(W2, X2, r)
        self.W, self.E = O.fold_vec(self.W, W2, r, p), O.fold_vec(self.E, T, r, p)
        self.X, self.u = O.fold_vec(self.X, X2, r, p), (self.u + r) % p

    def comm(self, v):
        return self.cv.msm_known_dlog(v, K0, D)

    def prove(self, tr=None):
        return self.rp.spartan_prove(self.gens, self.tau, tr or SR.Transcript())

    def accepts(self, pf, tr=None, comm_W=None) -> bool:
        """the verifier: transcript, both sum-checks with (A, B, C)(r_x, r_y) from the device, z(r_y) from eval_W and
        the public (u, X), and the opening under comm_E + rho comm_W by vdfgpu_ipa_verify_batch"""
        p, cv = self.p, self.cv
        if not SR.transcript_consistent(pf, tr or SR.Transcript(), p):
            return False
        if not SR.verify_claims(self.shape, self.u, self.X, self.tau, pf, self.gs.evaluate(pf.r_x, pf.r_y)):
            return False
        comm_W = self.comm(self.W) if comm_W is None else comm_W
        comm_a = cv.add(self.comm(self.E), cv.mul(pf.rho, comm_W))
        rs = [r for _, _, r in pf.ipa]
        b_hat = SP.ipa_b_hat(self.fid, rs, [(1, pf.r_x), (pf.rho, pf.r_y[1:])])
        proof = ([L for L, _, _ in pf.ipa], [R for _, R, _ in pf.ipa], rs, pf.a_hat, O.jac_to_bytes(cv, comm_a), pf.c,
                 b_hat, pf.u_scale)
        return SP.ipa_verify_batch(self.gens, [proof])[0]

    def close(self):
        self.rp.close()
        self.gs.close()
        self.gens.close()


# ---- parity and acceptance ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("fid", FIDS)
def test_parity_and_acceptance_on_a_folded_step(gpu_lib, fid):
    inst = Instance.folded_step(fid, 12, 100)
    assert inst.u != 1 and any(inst.E) and inst.shape.num_vars < inst.m
    pf = inst.prove()
    pts = inst.cv.progression(K0, D, inst.m + 1)
    assert pf == SR.prove(inst.shape, inst.W, inst.E, inst.u, inst.X, inst.tau, SR.Transcript(), inst.cv, pts)
    assert inst.accepts(pf)
    assert inst.gs.evaluate(pf.r_x, pf.r_y) == SR.evaluate(inst.shape, pf.r_x, pf.r_y)
    inst.close()


# ---- shapes ------------------------------------------------------------------------------------------------------
def _general(fid, cons, vars_, io):
    shape = S.general_shape(fid, cons, vars_, io)
    return Instance(fid, shape, *S.relaxed_instance(shape, seed=cons + vars_))


SHAPES = {
    "step t 30": lambda fid: Instance.folded_step(fid, 30, 0),
    "step t 20, aug 400": lambda fid: Instance.folded_step(fid, 20, 400),
    "general vars = m, io 2": lambda fid: _general(fid, 101, 128, 2),
    "general cons = m, io 0": lambda fid: _general(fid, 256, 150, 0),
    "general vars < cons, io 7": lambda fid: _general(fid, 333, 200, 7),
    "general vars > cons, io 7": lambda fid: _general(fid, 77, 300, 7),
}


@pytest.mark.parametrize("fid", FIDS)
@pytest.mark.parametrize("kind", sorted(SHAPES))
def test_shapes(gpu_lib, fid, kind):
    inst = SHAPES[kind](fid)
    if kind.startswith("general"):
        assert (inst.shape.num_vars > inst.shape.num_cons) == ("vars > cons" in kind or "vars = m" in kind)
    pf = inst.prove()
    assert inst.accepts(pf)
    assert inst.gs.evaluate(pf.r_x, pf.r_y) == SR.evaluate(inst.shape, pf.r_x, pf.r_y)
    inst.close()


def test_io_beyond_the_padded_size_is_an_argument_error(gpu_lib):
    p = O.Q
    shape = O.R1CSShape(p, 3, 2, 7, [(0, 0, 1)], [(1, 1, 1)], [(2, 9, 1)])   # m = 4 < 1 + 7
    inst = Instance(O.FIELD_FQ, shape, [1, 2], [0, 0, 0], 1, list(range(7)))
    with pytest.raises(VdfGpuError) as e:
        inst.rp.spartan_prove(inst.gens, [1, 2], SR.Transcript())
    assert e.value.code == -1
    with pytest.raises(VdfGpuError) as e:
        inst.gs.evaluate([1, 2], [1, 2, 3])
    assert e.value.code == -1
    inst.close()


# ---- rejection ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fid", FIDS)
def test_rejection(gpu_lib, fid):
    """one corrupted E entry: the call still proves, the verifier rejects; a wrong comm_W fails the opening"""
    inst = Instance.folded_step(fid, 12, 0)
    E = list(inst.E)
    E[7] = (E[7] + 1) % inst.p
    good = inst.prove()
    assert inst.accepts(good)
    assert not inst.accepts(good, comm_W=inst.cv.add(inst.comm(inst.W), inst.cv.gen))
    inst.set(inst.W, E, inst.u, inst.X)
    bad = inst.prove()
    assert not SR.verify_claims(inst.shape, inst.u, inst.X, inst.tau, bad, inst.gs.evaluate(bad.r_x, bad.r_y))
    inst.close()


# ---- the instance is left as it was -----------------------------------------------------------------------------
@pytest.mark.parametrize("fid", FIDS)
def test_instance_untouched(gpu_lib, fid):
    inst = Instance.folded_step(fid, 12, 50)
    before = inst.rp.get_running()
    assert before == (inst.W, inst.E, inst.u, inst.X)
    inst.prove()
    assert inst.rp.get_running() == before
    _, W3, X3, _ = O.make_step_instance(fid, 12, O.State(3, 4, 12), aug_cons=50)
    inst.fold(W3, X3, 0xABCDEF)
    assert inst.rp.get_running() == (inst.W, inst.E, inst.u, inst.X)
    inst.rp.U = N.RelaxedR1CSInstance(inst.comm(inst.W), inst.comm(inst.E), inst.X, inst.u)
    assert inst.rp.check().ok
    assert inst.accepts(inst.prove())
    inst.close()


# ---- ordering across streams -------------------------------------------------------------------------------------
def _delay(s, ms=25):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(torch.cuda.Stream()):
        a.record()
        torch.cuda._sleep(1_000_000)
        b.record()
    b.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(int(ms * 1_000_000 / max(a.elapsed_time(b), 1e-3)))


@pytest.mark.parametrize("prove_on", ["other stream", "same delayed stream"])
def test_prove_right_after_a_finish(gpu_lib, prove_on):
    """running_finish on stream A behind a delay returns at once; the prove on stream B (or on A itself) proves the
    folded instance"""
    import torch
    fid = O.FIELD_FQ
    inst = Instance.folded_step(fid, 12, 0)
    A, B = torch.cuda.Stream(), torch.cuda.Stream()
    _, W3, X3, _ = O.make_step_instance(fid, 12, O.State(3, 4, 12))
    try:
        _lib.check(gpu_lib.vdfgpu_set_stream(A.cuda_stream))
        T = inst.shape.cross_term(inst.W, inst.u, inst.X, W3, X3)
        cW, cT = bytearray(96), bytearray(96)
        _lib.check(gpu_lib.vdfgpu_running_commit(inst.rp._h, _lib.as_ptr(O.fes_to_bytes(W3, inst.p)),
                                                 _lib.as_ptr(O.fes_to_bytes(X3, inst.p)), _lib.as_ptr(cW),
                                                 _lib.as_ptr(cT)))
        _delay(A)
        r = 0x55AA
        _lib.check(gpu_lib.vdfgpu_running_finish(inst.rp._h, _lib.as_ptr(O.fe_to_bytes(r, inst.p))))
        p = inst.p
        inst.W, inst.E = O.fold_vec(inst.W, W3, r, p), O.fold_vec(inst.E, T, r, p)
        inst.X, inst.u = O.fold_vec(inst.X, X3, r, p), (inst.u + r) % p
        if prove_on == "other stream":
            _lib.check(gpu_lib.vdfgpu_set_stream(B.cuda_stream))
        pf = inst.prove()
        _lib.check(gpu_lib.vdfgpu_set_stream(None))
        assert inst.accepts(pf)
    finally:
        torch.cuda.synchronize()
        _lib.check(gpu_lib.vdfgpu_set_stream(None))
    inst.close()


# ---- two threads -------------------------------------------------------------------------------------------------
def test_primary_and_secondary_from_two_threads(gpu_lib):
    import torch
    insts = [Instance.folded_step(fid, 40, 200) for fid in FIDS]
    proofs, errors = [None, None], []

    def run(k):
        try:
            s = torch.cuda.Stream()
            _lib.check(gpu_lib.vdfgpu_set_stream(s.cuda_stream))
            proofs[k] = insts[k].prove(SR.Transcript(k))
            _lib.check(gpu_lib.vdfgpu_set_stream(None))
        except Exception as e:   # pragma: no cover - reported below
            errors.append(e)

    th = [threading.Thread(target=run, args=(k,)) for k in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errors, errors
    for k, inst in enumerate(insts):
        assert inst.accepts(proofs[k], SR.Transcript(k))
        inst.close()


# ---- errors ------------------------------------------------------------------------------------------------------
class Faulty(SR.Transcript):
    """SR.Transcript that misbehaves once, at `where`: raises, answers a non-canonical value (the modulus), or answers 0
    (an IPA challenge)"""
    WHERE = ["outer round", "OUTER", "inner round", "EVAL", "IPA", "ipa round"]

    def __init__(self, where, how, p, hook=None):
        super().__init__()
        self.where, self.how, self.p, self.hook = where, how, p, hook
        self.stages = 0

    def _bad(self, here, good):
        if here != self.where:
            return good
        if self.hook:
            self.hook()
            return good
        if self.how == "raise":
            raise RuntimeError("transcript failed")
        return self.p.to_bytes(32, "little") if self.how == "non-canonical" else 0

    def sumcheck_round(self, rnd, evals):
        here = "outer round" if self.stages == 0 else "inner round"
        return self._bad(here if rnd == 1 else None, super().sumcheck_round(rnd, evals))

    def claims(self, stage, values):
        self.stages += 1
        good = super().claims(stage, values)
        bad = self._bad(("OUTER", "EVAL", "IPA")[stage], None)
        return good if bad is None else [bad] + good[1:]

    def ipa_round(self, rnd, L, R):
        return self._bad("ipa round" if rnd == 1 else None, super().ipa_round(rnd, L, R))


@pytest.mark.parametrize("fid", FIDS)
def test_callback_failures(gpu_lib, fid):
    """each stage failing, or answering a non-canonical value, ends the call with VDFGPU_ERR_STATE; an IPA challenge
    of 0 too; the next call succeeds on the intact instance"""
    inst = Instance.folded_step(fid, 12, 0)
    good = inst.prove()
    for where in Faulty.WHERE:
        for how in ("raise", "non-canonical") + (("zero",) if where == "ipa round" else ()):
            with pytest.raises(VdfGpuError) as e:
                inst.prove(Faulty(where, how, inst.p))
            assert e.value.code == -3, (where, how)
            assert "running_spartan_prove" in str(e.value)
            assert inst.prove() == good, (where, how)
    assert inst.rp.get_running() == (inst.W, inst.E, inst.u, inst.X)
    inst.close()


def test_destroying_handles_during_a_call_is_refused(gpu_lib):
    inst = Instance.folded_step(O.FIELD_FQ, 12, 0)
    seen = []

    def destroy_all():
        seen.append((gpu_lib.vdfgpu_gens_destroy(inst.gens._h), gpu_lib.vdfgpu_r1cs_destroy(inst.gs._h),
                     gpu_lib.vdfgpu_running_destroy(inst.rp._h)))

    for where in Faulty.WHERE:
        pf = inst.prove(Faulty(where, None, inst.p, hook=destroy_all))
        assert inst.accepts(pf)
    assert seen == [(-3, -3, -3)] * len(Faulty.WHERE)
    inst.close()


def test_before_running_set_is_a_state_error(gpu_lib):
    shape, _, _, _ = O.make_step_instance(O.FIELD_FQ, 4, O.State(5, 6, 4))
    m = SR.padded_size(shape)
    gens = G.Generators.progression(O.CURVE_PALLAS, K0, D, m + 1)
    gs = N.R1CSShape(O.FIELD_FQ, shape.num_cons, shape.num_vars, shape.num_io, shape.A, shape.B, shape.C)
    rp = N.RunningProver(gs, gens)
    with pytest.raises(VdfGpuError) as e:
        rp.spartan_prove(gens, [1] * (m.bit_length() - 1), SR.Transcript())
    assert e.value.code == -3
    rp.close()
    gs.close()
    gens.close()


# ---- Nova sizes --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("t", [1024, 16384])
def test_nova_sizes(gpu_lib, t):
    """primary step shapes: every round by the O(ell) verifier, the claims against the oracle, the opening by
    vdfgpu_ipa_verify_batch"""
    inst = Instance.folded_step(O.FIELD_FQ, t, 0)
    pf = inst.prove()
    assert inst.accepts(pf)
    p, m = inst.p, inst.m
    eq_rx, eq_ry = O.eq_evals(pf.r_x, p), O.eq_evals(pf.r_y[1:], p)
    Cz = inst.shape.multiply_vec(inst.shape.z_of(inst.W, inst.u, inst.X))[2]
    dot = lambda a, b: sum(x * y for x, y in zip(a, b)) % p   # noqa: E731
    assert pf.outer_claims[2:] == (dot(Cz, eq_rx), dot(inst.E, eq_rx))
    assert pf.eval_claims == (dot(inst.W, eq_ry), (dot(inst.E, eq_ry) + dot(inst.W, eq_rx)) % p)
    assert len(pf.r_x) == m.bit_length() - 1
    inst.close()
