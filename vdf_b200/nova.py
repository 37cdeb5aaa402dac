"""Folding-side host interface: mirror of the nova-snark 0.8 types the reference drives through
RecursiveSNARK::prove_step (src/nova/proof.rs:342-349): R1CSShape::{multiply_vec, commit_T},
R1CSWitness::commit, RelaxedR1CS{Witness,Instance}::fold and NIFS::prove.  Vectors live on the GPU; this
module only marshals bytes and keeps the small instance data (u, X, commitments).

NOT mirrored (out of scope, SURVEY.md section 8): circuit synthesis (bellperson), the augmented circuit,
the Poseidon random oracle.  `challenge()` below is a labelled stand-in for the RO so that a chain of
fold steps can be driven end to end; swap it for nova's RO when binding from Rust (INTEGRATION.md).
"""
from __future__ import annotations

import ctypes
import hashlib
import struct
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

from . import _lib
from .encoding import (CURVE_BASE, CURVE_ORDER, CURVE_SCALAR_FIELD, MODULUS, POINT_BYTES, Affine,
                       affine_to_bytes, fe_to_bytes, fes_from_bytes, fes_to_bytes, point_from_bytes)
from .msm import Generators, mult_pippenger

Coo = List[Tuple[int, int, int]]  # (row, col, value)


def _coo_arrays(M: Coo, m: int):
    rows = struct.pack("<%dQ" % len(M), *[e[0] for e in M])
    cols = struct.pack("<%dQ" % len(M), *[e[1] for e in M])
    vals = fes_to_bytes([e[2] for e in M], m)
    return rows, cols, vals, len(M)


@dataclass
class SatReport:
    """Verdict of one satisfiability check (RelaxedR1CSShape::is_sat_relaxed / R1CSShape::is_sat): the rows where
    Az.Bz != u.Cz + E, and whether each commitment equals the commitment of its vector (None: not checked)."""
    bad_rows: int
    first_bad_row: Optional[int]
    comm_W_ok: Optional[bool]
    comm_E_ok: Optional[bool]

    @property
    def ok(self) -> bool:
        return self.bad_rows == 0 and self.comm_W_ok is not False and self.comm_E_ok is not False

    @classmethod
    def from_words(cls, rep, num_cons: int) -> "SatReport":
        verdict = {0: False, 1: True, 2: None}
        return cls(int(rep[0]), None if rep[1] == num_cons else int(rep[1]), verdict[rep[2]], verdict[rep[3]])


def _point_arg(p, base: int) -> Optional[bytes]:
    """A commitment as the 96-byte Jacobian point the C ABI compares: an affine tuple, or 96 raw bytes (any Z, the
    identity as Z = 0).  None: not checked."""
    if p is None:
        return None
    if isinstance(p, (bytes, bytearray)):
        if len(p) != POINT_BYTES:
            raise ValueError("a commitment is a 96-byte Jacobian point")
        return bytes(p)
    return fe_to_bytes(p[0], base) + fe_to_bytes(p[1], base) + fe_to_bytes(1, base)


class R1CSShape:
    """nova R1CSShape: A, B, C in COO over z = [W | u | X]; uploaded once as CSR."""

    def __init__(self, field_id: int, num_cons: int, num_vars: int, num_io: int, A: Coo, B: Coo, C: Coo):
        self.field_id = field_id
        self.m = MODULUS[field_id]
        self.num_cons, self.num_vars, self.num_io = num_cons, num_vars, num_io
        self.nnz = len(A) + len(B) + len(C)
        a, b, c = (_coo_arrays(M, self.m) for M in (A, B, C))
        h = ctypes.c_void_p()
        _lib.check(_lib.load().vdfgpu_r1cs_create(
            field_id, num_cons, num_vars, num_io,
            _lib.as_ptr(a[0]), _lib.as_ptr(a[1]), _lib.as_ptr(a[2]), a[3],
            _lib.as_ptr(b[0]), _lib.as_ptr(b[1]), _lib.as_ptr(b[2]), b[3],
            _lib.as_ptr(c[0]), _lib.as_ptr(c[1]), _lib.as_ptr(c[2]), c[3], ctypes.byref(h)))
        self._h = h

    def multiply_vec(self, z: Sequence[int]) -> Tuple[List[int], List[int], List[int]]:
        if len(z) != self.num_vars + 1 + self.num_io:
            raise ValueError("z has the wrong length")  # nova: NovaError::InvalidWitnessLength
        outs = [bytearray(self.num_cons * 32) for _ in range(3)]
        _lib.check(_lib.load().vdfgpu_multiply_vec(self._h, _lib.as_ptr(fes_to_bytes(z, self.m)),
                                                   *[_lib.as_ptr(o) for o in outs]))
        return tuple(fes_from_bytes(bytes(o), self.m) for o in outs)

    def bind_rows(self, eq_rows: Sequence[int], r_abc: Sequence[int]) -> List[int]:
        """Spartan's inner sum-check table: out[y] = sum_x eq_rows[x] (rA A[x,y] + rB B[x,y] + rC C[x,y])
        (nova-snark compute_eval_table_sparse + the three challenges; CompressedSNARK::prove, src/nova/proof.rs:363)."""
        if len(eq_rows) != self.num_cons or len(r_abc) != 3:
            raise ValueError("eq_rows needs one entry per constraint and r_abc three challenges")
        out = bytearray((self.num_vars + 1 + self.num_io) * 32)
        _lib.check(_lib.load().vdfgpu_r1cs_bind_rows(self._h, _lib.as_ptr(fes_to_bytes(eq_rows, self.m)),
                                                     _lib.as_ptr(fes_to_bytes(r_abc, self.m)), _lib.as_ptr(out)))
        return fes_from_bytes(bytes(out), self.m)

    def evaluate(self, rx: Sequence[int], ry: Sequence[int]) -> Tuple[int, int, int]:
        """(A, B, C)(r_x, r_y) over nova's padded layout (spartan.padded_layout): the sparse evaluation of
        RelaxedR1CSSNARK::verify [R].  rx: log2 m coordinates, ry: log2 m + 1, most significant variable first."""
        from .spartan import padded_layout
        m, _ = padded_layout(self.num_cons, self.num_vars, self.num_io)
        ell_x = m.bit_length() - 1
        if len(rx) != ell_x or len(ry) != ell_x + 1:
            raise ValueError("evaluate: rx needs log2 m coordinates and ry one more")
        out = bytearray(96)
        _lib.check(_lib.load().vdfgpu_r1cs_evaluate(self._h, _lib.as_ptr(fes_to_bytes(rx, self.m) or bytes(32)),
                                                    _lib.as_ptr(fes_to_bytes(ry, self.m)), _lib.as_ptr(out)))
        return tuple(fes_from_bytes(bytes(out), self.m))

    def evaluate_batch(self, rxs: Sequence[Sequence[int]], rys: Sequence[Sequence[int]]) -> List[Tuple[int, int, int]]:
        """evaluate at k points in one pass (vdfgpu_r1cs_evaluate_batch): one (A, B, C) per (rx, ry) pair."""
        from .spartan import padded_layout
        m, _ = padded_layout(self.num_cons, self.num_vars, self.num_io)
        ell_x = m.bit_length() - 1
        k = len(rxs)
        if k == 0 or len(rys) != k or any(len(rx) != ell_x for rx in rxs) or any(len(ry) != ell_x + 1 for ry in rys):
            raise ValueError("evaluate_batch: k >= 1 points, each rx with log2 m coordinates and ry with one more")
        out = bytearray(96 * k)
        _lib.check(_lib.load().vdfgpu_r1cs_evaluate_batch(
            self._h, k, _lib.as_ptr(fes_to_bytes([v for rx in rxs for v in rx], self.m) or bytes(32)),
            _lib.as_ptr(fes_to_bytes([v for ry in rys for v in ry], self.m)), _lib.as_ptr(out)))
        vals = fes_from_bytes(bytes(out), self.m)
        return [tuple(vals[3 * q:3 * q + 3]) for q in range(k)]

    def commit_T(self, gens: Optional[Generators], W1: Sequence[int], u1: int, X1: Sequence[int],
                 W2: Sequence[int], X2: Sequence[int]) -> Tuple[List[int], Affine]:
        """Cross-term T and its commitment (u2 = 1 for the fresh instance)."""
        T = bytearray(self.num_cons * 32)
        comm = bytearray(POINT_BYTES)
        m = self.m
        _lib.check(_lib.load().vdfgpu_commit_T(
            self._h, gens._h if gens else None, _lib.as_ptr(fes_to_bytes(W1, m)), _lib.as_ptr(fe_to_bytes(u1, m)),
            _lib.as_ptr(fes_to_bytes(X1, m)), _lib.as_ptr(fes_to_bytes(W2, m)), _lib.as_ptr(fes_to_bytes(X2, m)),
            _lib.as_ptr(T), _lib.as_ptr(comm) if gens else None))
        cT = point_from_bytes(bytes(comm), CURVE_BASE[gens.curve]) if gens else None
        return fes_from_bytes(bytes(T), m), cT

    def is_sat_relaxed(self, gens: Optional[Generators], W: Sequence[int], E: Optional[Sequence[int]],
                       U: "RelaxedR1CSInstance") -> SatReport:
        """RelaxedR1CSShape::is_sat_relaxed: Az.Bz = u.Cz + E on every row, comm_W = commit(W), comm_E = commit(E).
        E None means E = 0; a commitment of U that is None is not checked (gens None: neither is)."""
        if len(W) != self.num_vars or len(U.X) != self.num_io or (E is not None and len(E) != self.num_cons):
            raise ValueError("W, E or X has the wrong length")  # nova: NovaError::InvalidWitnessLength
        m = self.m
        return self._check(gens, fes_to_bytes(W, m), None if E is None else fes_to_bytes(E, m), fe_to_bytes(U.u, m),
                           fes_to_bytes(U.X, m), U.comm_W, U.comm_E)

    def is_sat(self, gens: Optional[Generators], W: Sequence[int], X: Sequence[int], comm_W=None) -> SatReport:
        """R1CSShape::is_sat of a fresh instance: Az.Bz = Cz (u = 1, E = 0) and comm_W = commit(W)."""
        if len(W) != self.num_vars or len(X) != self.num_io:
            raise ValueError("W or X has the wrong length")  # nova: NovaError::InvalidWitnessLength
        m = self.m
        return self._check(gens, fes_to_bytes(W, m), None, None, fes_to_bytes(X, m), comm_W, None)

    def _check(self, gens, Wb, Eb, ub, Xb, comm_W, comm_E) -> SatReport:
        if gens is None and (comm_W is not None or comm_E is not None):
            raise ValueError("checking a commitment needs the generators")
        cW, cE = (_point_arg(c, CURVE_BASE[gens.curve]) if gens else None for c in (comm_W, comm_E))
        rep = (ctypes.c_uint64 * 4)()
        _lib.check(_lib.load().vdfgpu_r1cs_is_sat_relaxed(
            self._h, gens._h if gens else None, _lib.as_ptr(Wb), _lib.as_ptr(Eb), _lib.as_ptr(ub), _lib.as_ptr(Xb),
            _lib.as_ptr(cW), _lib.as_ptr(cE), rep))
        return SatReport.from_words(rep, self.num_cons)

    def is_sat_relaxed_dev(self, W_dev, E_dev, uX_dev, counts2_dev) -> None:
        """Row check on device buffers (torch tensors or raw pointers), enqueued on the calling thread's stream:
        counts2_dev receives (violating rows, smallest violating row or num_cons) as two u64."""
        _lib.check(_lib.load().vdfgpu_r1cs_is_sat_relaxed_dev(self._h, _lib.as_ptr(W_dev), _lib.as_ptr(E_dev),
                                                              _lib.as_ptr(uX_dev), _lib.as_ptr(counts2_dev)))

    def close(self):
        if self._h:
            _lib.load().vdfgpu_r1cs_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def fold_vectors(field_id: int, W1: Sequence[int], W2: Sequence[int], E1: Sequence[int], T: Sequence[int], r: int):
    """RelaxedR1CSWitness::fold on host vectors: (W1 + r W2, E1 + r T)."""
    m = MODULUS[field_id]
    w = bytearray(fes_to_bytes(W1, m))
    e = bytearray(fes_to_bytes(E1, m))
    _lib.check(_lib.load().vdfgpu_fold(field_id, _lib.as_ptr(w), _lib.as_ptr(fes_to_bytes(W2, m)), len(W1),
                                       _lib.as_ptr(e), _lib.as_ptr(fes_to_bytes(T, m)), len(E1),
                                       _lib.as_ptr(fe_to_bytes(r, m))))
    return fes_from_bytes(bytes(w), m), fes_from_bytes(bytes(e), m)


def point_fold(curve: int, P1: Affine, P2: Affine, r: int) -> Affine:
    """P1 + r * P2 (RelaxedR1CSInstance::fold's commitment update) as a 2-point MSM on the GPU."""
    base, order = CURVE_BASE[curve], CURVE_ORDER[curve]
    pts = affine_to_bytes(P1, base) + affine_to_bytes(P2, base)
    sc = fe_to_bytes(1, order) + fe_to_bytes(r, order)
    return point_from_bytes(mult_pippenger(curve, pts, sc, True), base)


def challenge(*chunks: bytes) -> int:
    """STAND-IN for nova's Poseidon random oracle: 128-bit challenge from BLAKE2b of the transcript."""
    h = hashlib.blake2b(digest_size=16)
    for c in chunks:
        h.update(c)
    return int.from_bytes(h.digest(), "little")


class WitnessBank:
    """Step-circuit witnesses (4t+1 values per step, src/nova/proof.rs:107-126, :162-189) of all steps of a proof,
    generated and kept on the device (SURVEY.md section 8f rank 1).  `states` are the steps' input states (x, y, i)."""

    def __init__(self, field_id: int, states: Sequence[Tuple[int, int, int]], t: int):
        m = MODULUS[field_id]
        self.field_id, self.t, self.n, self.m = field_id, t, len(states), m
        raw = b"".join(fes_to_bytes(list(s), m) for s in states)
        h = ctypes.c_void_p()
        _lib.check(_lib.load().vdfgpu_witness_bank_create(field_id, _lib.as_ptr(raw), t, len(states), ctypes.byref(h)))
        self._h = h

    def read(self, first: int = 0, count: Optional[int] = None) -> List[List[int]]:
        count = self.n - first if count is None else count
        per = 4 * self.t + 1
        buf = bytearray(count * per * 32)
        _lib.check(_lib.load().vdfgpu_witness_bank_read(self._h, first, count, _lib.as_ptr(buf)))
        flat = fes_from_bytes(bytes(buf), self.m)
        return [flat[k * per:(k + 1) * per] for k in range(count)]

    def close(self):
        if self._h:
            _lib.load().vdfgpu_witness_bank_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


@dataclass
class RelaxedR1CSInstance:  # nova RelaxedR1CSInstance
    comm_W: Affine
    comm_E: Affine
    X: List[int]
    u: int


@dataclass
class SpartanProof:
    """What vdfgpu_running_spartan_prove handed to the transcript, in order (RelaxedR1CSSNARK::prove [R]): the outer
    sum-check's rounds ((e0, e2, e3), r), the OUTER claims (claim_Az, claim_Bz, claim_Cz, eval_E) and (r_A, r_B, r_C),
    the inner rounds ((e0, e2), r), the EVAL claims (eval_W, T) and rho, the joint claim c and u_scale, the IPA's
    (L, R, r) with L and R as 96-byte normalised points, and a_hat."""
    outer: List[Tuple[Tuple[int, ...], int]]
    outer_claims: Tuple[int, ...]
    r_abc: Tuple[int, ...]
    inner: List[Tuple[Tuple[int, ...], int]]
    eval_claims: Tuple[int, ...]
    rho: int
    c: int
    u_scale: int
    ipa: List[Tuple[bytes, bytes, int]]
    a_hat: int

    @property
    def r_x(self) -> List[int]:
        return [r for _, r in self.outer]

    @property
    def r_y(self) -> List[int]:
        return [r for _, r in self.inner]

    @classmethod
    def from_log(cls, log: list, a_hat: int) -> "SpartanProof":
        rounds = [[], []]
        claims = {}
        for e in log:
            if e[0] == "round":
                rounds[1 if claims else 0].append((e[1], e[2]))
            elif e[0] == "claims":
                claims[e[1]] = (e[2], e[3])
        (oc, rabc), (ev, rho), (c, us) = (claims[k] for k in range(3))
        return cls(rounds[0], oc, rabc, rounds[1], ev, rho[0], c[0], us[0],
                   [(e[1], e[2], e[3]) for e in log if e[0] == "ipa"], a_hat)


@dataclass
class RunningProver:
    """Device-resident running (W, E) for one curve + the instance on the host: NIFS::prove per step."""
    shape: R1CSShape
    gens: Generators
    U: RelaxedR1CSInstance = None
    _h: ctypes.c_void_p = field(default_factory=ctypes.c_void_p)

    def __post_init__(self):
        h = ctypes.c_void_p()
        _lib.check(_lib.load().vdfgpu_running_create(self.shape._h, self.gens._h, ctypes.byref(h)))
        self._h = h

    def set_running(self, W: Sequence[int], E: Sequence[int], U: RelaxedR1CSInstance) -> None:
        m = self.shape.m
        _lib.check(_lib.load().vdfgpu_running_set(self._h, _lib.as_ptr(fes_to_bytes(W, m)), _lib.as_ptr(fes_to_bytes(E, m)),
                                                  _lib.as_ptr(fe_to_bytes(U.u, m)), _lib.as_ptr(fes_to_bytes(U.X, m))))
        self.U = U

    def get_running(self) -> Tuple[List[int], List[int], int, List[int]]:
        s = self.shape
        W, E = bytearray(s.num_vars * 32), bytearray(s.num_cons * 32)
        u, X = bytearray(32), bytearray(max(1, s.num_io) * 32)
        _lib.check(_lib.load().vdfgpu_running_get(self._h, _lib.as_ptr(W), _lib.as_ptr(E), _lib.as_ptr(u), _lib.as_ptr(X)))
        m = s.m
        return (fes_from_bytes(bytes(W), m), fes_from_bytes(bytes(E), m), fes_from_bytes(bytes(u), m)[0],
                fes_from_bytes(bytes(X[:s.num_io * 32]), m))

    def check(self) -> SatReport:
        """is_sat_relaxed of the resident running instance against self.U's commitments (None: not checked); W, E,
        u and X stay on the device."""
        base = CURVE_BASE[self.gens.curve]
        cW, cE = (_point_arg(c, base) for c in ((self.U.comm_W, self.U.comm_E) if self.U else (None, None)))
        rep = (ctypes.c_uint64 * 4)()
        _lib.check(_lib.load().vdfgpu_running_check(self._h, _lib.as_ptr(cW), _lib.as_ptr(cE), rep))
        return SatReport.from_words(rep, self.shape.num_cons)

    def spartan_prove(self, ipa_gens: Generators, tau: Sequence[int], transcript) -> SpartanProof:
        """RelaxedR1CSSNARK::prove [R] of the resident running instance in one call (vdfgpu_running_spartan_prove):
        W, E, u and X are not read back.  ipa_gens: at least m + 1 points of this curve, the first m the commitment
        generators.  tau: log2 m elements.  transcript: an object with sumcheck_round(rnd, evals), claims(stage, values)
        and ipa_round(rnd, L, R), each returning an integer (or 32 raw bytes); see include/vdfgpu.h for what each stage
        receives and returns."""
        from .spartan import padded_layout, spartan_trampolines
        s = self.shape
        m_pad, _ = padded_layout(s.num_cons, s.num_vars, s.num_io)
        if len(tau) != m_pad.bit_length() - 1:
            raise ValueError("spartan_prove: tau needs log2 m elements")
        log: list = []
        cbs = spartan_trampolines(s.m, transcript, log)
        a_hat = bytearray(32)
        _lib.check(_lib.load().vdfgpu_running_spartan_prove(
            self._h, ipa_gens._h, _lib.as_ptr(fes_to_bytes(tau, s.m) or bytes(32)),
            *[ctypes.cast(cb, ctypes.c_void_p) for cb in cbs], None, _lib.as_ptr(a_hat)))
        return SpartanProof.from_log(log, fes_from_bytes(bytes(a_hat), s.m)[0])

    def prove_step_bytes(self, W2: bytes, X2: bytes, r: Optional[int] = None):
        """One fold of a fresh satisfying (W2, X2): returns (comm_W2, comm_T, r) with points as 96-byte
        buffers.  Timed region of the fold-steps/s benchmark."""
        lib = _lib.load()
        cW, cT = bytearray(POINT_BYTES), bytearray(POINT_BYTES)
        _lib.check(lib.vdfgpu_running_commit(self._h, _lib.as_ptr(W2), _lib.as_ptr(X2), _lib.as_ptr(cW), _lib.as_ptr(cT)))
        if r is None:
            # the transcript absorbs canonical (affine) encodings, as nova's RO does via to_affine()
            base = CURVE_BASE[self.gens.curve]
            r = challenge(*[affine_to_bytes(point_from_bytes(bytes(c), base), base) for c in (cW, cT)])
        _lib.check(lib.vdfgpu_running_finish(self._h, _lib.as_ptr(fe_to_bytes(r, self.shape.m))))
        return bytes(cW), bytes(cT), r

    def prove_step_bank_bytes(self, bank: WitnessBank, step: int, step_offset: int, W2: bytes, X2: bytes, r: int):
        """prove_step_bytes with the 4t+1 step variables of W2 taken from the device-resident bank: the bytes of
        W2[step_offset : step_offset + 4t + 1] are ignored and never transferred."""
        lib = _lib.load()
        cW, cT = bytearray(POINT_BYTES), bytearray(POINT_BYTES)
        _lib.check(lib.vdfgpu_running_commit_step(self._h, bank._h, step, step_offset, _lib.as_ptr(W2), _lib.as_ptr(X2),
                                                  _lib.as_ptr(cW), _lib.as_ptr(cT)))
        _lib.check(lib.vdfgpu_running_finish(self._h, _lib.as_ptr(fe_to_bytes(r, self.shape.m))))
        return bytes(cW), bytes(cT), r

    def prove_step(self, W2: Sequence[int], X2: Sequence[int], r: Optional[int] = None):
        """NIFS::prove against the running instance: commit(W2), commit_T, challenge, fold witness and
        instance.  Returns (comm_T, r)."""
        m = self.shape.m
        curve = self.gens.curve
        base = CURVE_BASE[curve]
        cW, cT, r = self.prove_step_bytes(fes_to_bytes(W2, m), fes_to_bytes(X2, m), r)
        comm_W2, comm_T = point_from_bytes(cW, base), point_from_bytes(cT, base)
        U = self.U
        self.U = RelaxedR1CSInstance(
            comm_W=point_fold(curve, U.comm_W, comm_W2, r),
            comm_E=point_fold(curve, U.comm_E, comm_T, r),
            X=[(a + r * b) % m for a, b in zip(U.X, X2)],
            u=(U.u + r) % m)
        return comm_T, r

    def close(self):
        if self._h:
            _lib.load().vdfgpu_running_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class RecursiveProver:
    """The GPU side of RecursiveSNARK::prove_step (src/nova/proof.rs:342-349) for BOTH curves of the cycle: per fold
    step NIFS::prove on the secondary curve (Vesta: the instance produced by the previous step's secondary circuit is
    folded into the secondary running instance), then NIFS::prove on the primary curve (Pallas: the step circuit's
    fresh instance).  The two are strictly sequential -- the primary circuit's public input hashes the secondary
    fold's output -- so this object only owns the two device-resident running instances and drives them in that
    order; synthesis of the augmented circuits and the random oracle stay on the host (`challenge` is the labelled
    stand-in)."""

    def __init__(self, primary: RunningProver, secondary: RunningProver):
        self.primary, self.secondary = primary, secondary
        self.steps = 0

    def prove_step(self, sec_W2: Sequence[int], sec_X2: Sequence[int], pri_W2: Sequence[int], pri_X2: Sequence[int],
                   r_sec: Optional[int] = None, r_pri: Optional[int] = None):
        """One fold step; returns ((comm_T_sec, r_sec), (comm_T_pri, r_pri))."""
        a = self.secondary.prove_step(sec_W2, sec_X2, r_sec)
        b = self.primary.prove_step(pri_W2, pri_X2, r_pri)
        self.steps += 1
        return a, b

    def prove_step_bytes(self, sec_W2: bytes, sec_X2: bytes, pri_W2: bytes, pri_X2: bytes, r_sec: int, r_pri: int,
                         bank: Optional[WitnessBank] = None, step: int = 0, step_offset: int = 0):
        """Byte-level form (the timed region of the fold-steps/s benchmark).  With `bank`, the 4t+1 step variables of
        the primary witness come from the device-resident witness bank."""
        a = self.secondary.prove_step_bytes(sec_W2, sec_X2, r_sec)
        if bank is None:
            b = self.primary.prove_step_bytes(pri_W2, pri_X2, r_pri)
        else:
            b = self.primary.prove_step_bank_bytes(bank, step, step_offset, pri_W2, pri_X2, r_pri)
        self.steps += 1
        return a, b

    def check(self) -> Tuple[SatReport, SatReport]:
        """is_sat_relaxed of the primary and the secondary running instance (RecursiveSNARK::verify's two relaxed
        checks, src/nova/proof.rs:382), on the device-resident vectors."""
        return self.primary.check(), self.secondary.check()

