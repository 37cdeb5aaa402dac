"""GPU: Spartan proofs verified in batches (vdfgpu_spartan_verify_batch) and the batched sparse evaluation
(vdfgpu_r1cs_evaluate_batch), both fields/curves, on proofs from vdfgpu_running_spartan_prove: acceptance with every
verdict equal to the per-proof verifier of tests/test_gpu_spartan.py; one corruption at a time in one proof of a batch;
malformed proofs as verdicts; the weights; parity of the batched evaluation with single calls and tests/spartan_ref.py;
Nova sizes; two threads on their own streams."""
import random
import threading

import pytest

from oracle import pasta as O
from tests import spartan_ref as SR
from tests import spartan_verify_ref as SVR
from tests.test_gpu_spartan import D, FIDS, K0, SHAPES, Instance
from vdf_b200 import _lib
from vdf_b200 import spartan as SP

pytestmark = pytest.mark.gpu


def _items(inst, k, salt0=0):
    """k proofs of the instance under k transcripts, as (item, transcript) pairs"""
    cW, cE = inst.comm(inst.W), inst.comm(inst.E)
    out = []
    for salt in range(salt0, salt0 + k):
        tr = SR.Transcript(salt)
        out.append(((inst.u, inst.X, cW, cE, inst.tau, inst.prove(tr)), tr))
    return out


def _verify(inst, items, weights=None):
    return SP.spartan_verify_batch(inst.gs, inst.gens, items, weights)


# ---- acceptance ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fid", FIDS)
@pytest.mark.parametrize("kind", sorted(SHAPES))
@pytest.mark.parametrize("k", [1, 5])
def test_acceptance(gpu_lib, fid, kind, k):
    inst = SHAPES[kind](fid)
    pairs = _items(inst, k)
    got = _verify(inst, [it for it, _ in pairs])
    assert got == [True] * k
    assert got == [inst.accepts(it[5], tr) for it, tr in pairs]
    inst.close()


# ---- one corruption at a time --------------------------------------------------------------------------------------
@pytest.mark.parametrize("fid", FIDS)
def test_one_corrupted_proof_of_a_batch(gpu_lib, fid):
    """exactly the corrupted proof is rejected, the others accepted, for every corruption; the per-proof verifier
    agrees"""
    inst = Instance.folded_step(fid, 12, 50)
    items = [it for it, _ in _items(inst, 3)]
    for what in SVR.CORRUPTIONS:
        bad = list(items)
        bad[1] = SVR.corrupt(items[1], what, inst.cv, inst.p)
        assert _verify(inst, bad) == [True, False, True], what
        if what not in ("u", "X", "comm_E", "r_y[0]"):   # the instance and transcript of Instance.accepts are fixed
            assert not inst.accepts(bad[1][5], SR.Transcript(1), comm_W=bad[1][2]), what
    inst.close()


# ---- malformed proofs ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fid", FIDS)
def test_malformed_proofs_are_verdicts(gpu_lib, fid):
    """an off-curve comm_E, a coordinate >= p, a non-canonical claim: verdict 0 for that proof only"""
    inst = Instance.folded_step(fid, 12, 0)
    items = [it for it, _ in _items(inst, 4)]
    ell = inst.m.bit_length() - 1
    PF, NP = 5 * ell + 9, 2 * ell + 2
    base = inst.cv.base
    inst_b, pts, proof, chal = SP.spartan_records(inst.gs, inst.gens.curve, items)
    at = 96 * (0 * NP + 1)                                     # proof 0: comm_E off the curve
    y = O.fe_from_bytes(pts[at + 32:at + 64], base)
    pts = pts[:at + 32] + O.fe_to_bytes(y + 1, base) + pts[at + 64:]
    at = 96 * (2 * NP)                                         # proof 2: comm_W.X = p
    pts = pts[:at] + base.to_bytes(32, "little") + pts[at + 32:]
    at = 32 * (3 * PF + 3 * ell + 2)                           # proof 3: claim_Cz = the modulus
    proof = proof[:at] + inst.p.to_bytes(32, "little") + proof[at + 32:]
    assert SP.spartan_verify_records(inst.gs, inst.gens, 4, inst_b, pts, proof, chal) == [False, True, False, False]
    inst.close()


# ---- weights -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fid", FIDS)
def test_weights_must_be_random(gpu_lib, fid):
    """two openings whose errors cancel under w = (1, 1) pass with those weights and are caught with random ones"""
    inst = Instance.folded_step(fid, 12, 0)
    a, b = (list(it) for it, _ in _items(inst, 2))
    d = inst.cv.mul(987654321, inst.cv.gen)
    a[3], b[3] = inst.cv.add(a[3], d), inst.cv.add(b[3], inst.cv.neg(d))
    pair = [tuple(a), tuple(b)]
    assert _verify(inst, pair, [1, 1]) == [True, True]
    assert _verify(inst, pair) == [False, False]
    inst.close()


# ---- the batched evaluation ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("fid", FIDS)
@pytest.mark.parametrize("kind", sorted(k for k in SHAPES if k.startswith("general")))
def test_evaluate_batch_parity(gpu_lib, fid, kind):
    """k = 1, 3, 64: equal to k calls of vdfgpu_r1cs_evaluate and to spartan_ref.evaluate"""
    inst = SHAPES[kind](fid)
    p = inst.p
    ell = inst.m.bit_length() - 1
    py = random.Random(ell * 31 + fid)
    for k in (1, 3, 64):
        rxs = [[py.randrange(p) for _ in range(ell)] for _ in range(k)]
        rys = [[py.randrange(p) for _ in range(ell + 1)] for _ in range(k)]
        got = inst.gs.evaluate_batch(rxs, rys)
        assert got == [inst.gs.evaluate(rx, ry) for rx, ry in zip(rxs, rys)]
        sample = range(k) if k <= 3 else range(0, k, 9)
        assert [got[q] for q in sample] == [SR.evaluate(inst.shape, rxs[q], rys[q]) for q in sample]
    inst.close()


def test_evaluate_batch_at_nova_size(gpu_lib):
    """t = 16 384 step shape, k = 8 random points: equal to eight single calls"""
    from vdf_b200 import nova as N
    fid = O.FIELD_FQ
    shape, _, _, _ = O.make_step_instance(fid, 16384, O.State(5, 6, 16384))
    gs = N.R1CSShape(fid, shape.num_cons, shape.num_vars, shape.num_io, shape.A, shape.B, shape.C)
    ell = SR.padded_size(shape).bit_length() - 1
    py = random.Random(8)
    rxs = [[py.randrange(shape.m) for _ in range(ell)] for _ in range(8)]
    rys = [[py.randrange(shape.m) for _ in range(ell + 1)] for _ in range(8)]
    assert gs.evaluate_batch(rxs, rys) == [gs.evaluate(rx, ry) for rx, ry in zip(rxs, rys)]
    gs.close()


# ---- Nova sizes ----------------------------------------------------------------------------------------------------
def _synthetic(fid, t, aug, seed):
    """a satisfied relaxed instance (u != 1, dense E) of bench.py's step shapes"""
    from vdf_b200 import synthetic as SY
    cons, nv, io, A, B, C, W, X = SY.step_instance(fid, t, aug, seed=seed)
    shape = O.R1CSShape(O.MODULUS[fid], cons, nv, io, A, B, C)
    u = 0x1234567890ABCDEF1234567890ABCDEF
    Az, Bz, Cz = shape.multiply_vec(shape.z_of(W, u, X))
    p = shape.m
    E = [(a * b - u * c) % p for a, b, c in zip(Az, Bz, Cz)]
    return Instance(fid, shape, W, E, u, X)


@pytest.mark.parametrize("side", ["primary t 1024", "primary t 16384", "secondary"])
def test_nova_sizes(gpu_lib, side):
    """four proofs each, all accepted; one corrupted proof rejected"""
    inst = {"primary t 1024": lambda: _synthetic(O.FIELD_FQ, 1024, 9800, 42),
            "primary t 16384": lambda: _synthetic(O.FIELD_FQ, 16384, 9800, 42),
            "secondary": lambda: _synthetic(O.FIELD_FP, 0, 10300, 7)}[side]()
    items = [it for it, _ in _items(inst, 4)]
    assert _verify(inst, items) == [True] * 4
    bad = list(items)
    bad[2] = SVR.corrupt(items[2], "inner round", inst.cv, inst.p)
    assert _verify(inst, bad) == [True, True, False, True]
    inst.close()


# ---- two threads ---------------------------------------------------------------------------------------------------
def test_two_threads_on_their_own_streams(gpu_lib):
    import torch
    insts = [Instance.folded_step(fid, 40, 200) for fid in FIDS]
    batches = [[it for it, _ in _items(inst, 3, 10 * n)] for n, inst in enumerate(insts)]
    batches[1][1] = SVR.corrupt(batches[1][1], "eval_W", insts[1].cv, insts[1].p)
    results, errors = [None, None], []

    def run(n):
        try:
            s = torch.cuda.Stream()
            _lib.check(gpu_lib.vdfgpu_set_stream(s.cuda_stream))
            for _ in range(3):
                results[n] = _verify(insts[n], batches[n])
            _lib.check(gpu_lib.vdfgpu_set_stream(None))
        except Exception as e:   # pragma: no cover - reported below
            errors.append(e)

    th = [threading.Thread(target=run, args=(n,)) for n in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errors, errors
    assert results == [[True, True, True], [True, False, True]]
    for inst in insts:
        inst.close()
