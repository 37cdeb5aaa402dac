#!/usr/bin/env python
"""RelaxedR1CSSNARK::verify of k proofs in one call (vdfgpu_spartan_verify_batch) at the step shapes of bench.py:
primary (Pallas, t = 10, 1024, 16384, SYNTHETIC 9.8k-constraint augmented block) and secondary (Vesta, SYNTHETIC
10.3k-constraint augmented circuit).  The proofs are k distinct proofs of one satisfied relaxed instance (u != 1, dense
E) from vdfgpu_running_spartan_prove under k sha256 transcripts; the IPA set is a table-layout progression of m + 1
points.  Per shape and k = 1, 8, 64:
  call_ms        wall time of one call with its records encoded beforehand, ending in the library's wait; median of
                 --runs after --warm
  composed_ms    what the call replaces, in the same run: k x vdfgpu_r1cs_evaluate, then one vdfgpu_ipa_verify_batch with
                 comm_E + rho comm_W, c and b_hat formed beforehand (the host sum-check checks are left out, which
                 favours this path)
  kernels_us     device time per call of the batched evaluation's kernels (torch.profiler kernel records, a pass of its
                 own): sparse_eval_batch_kernel, the half tables (EqHalfTablesBatchFn) and the column sums
  mults          field multiplications of sparse_eval_batch_kernel per call: k (nnz (1 + f) + 4 cons), f the share of
                 coefficients other than +-1; mul_per_s and the fraction of the multiplier's 7.6e10 mul/s
At k = 64 also host_ms: torch.profiler CPU timestamps from the call's start to its first runtime call that enqueues
device work (the argument and host checks, and the opening's point checks).  Writes one JSON line (default
profiles/r4_spartan_verify.json) with the device name, power limit and max SM clock read in the same run."""
import argparse
import json
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from profile_ipa_verify import DEVICE_WORK, stats   # noqa: E402

K0, D = 1234567, 89
MUL_RATE = 7.6e10   # DESIGN.md section 2.1: the field multiplier's measured rate on the B200


def side(fid, cid, t, aug, seed, kmax):
    from oracle import pasta as O
    from tests import spartan_ref as SR
    from vdf_b200 import encoding as E, msm as G, nova as N, synthetic as S
    from vdf_b200.spartan import padded_layout
    cons, nvars, io, A, B, Cm, W, X = S.step_instance(fid, t, aug, seed=seed)
    p = E.MODULUS[fid]
    gs = N.R1CSShape(fid, cons, nvars, io, A, B, Cm)
    m, _ = padded_layout(cons, nvars, io)
    gens = G.Generators.progression(cid, K0, D, m + 1, table=True)
    u = 0x1234567890ABCDEF1234567890ABCDEF
    Az, Bz, Cz = gs.multiply_vec(list(W) + [u] + list(X))
    Er = [(a * b - u * c) % p for a, b, c in zip(Az, Bz, Cz)]
    pr = N.RunningProver(gs, gens)
    pr.set_running(W, Er, N.RelaxedR1CSInstance(None, None, list(X), u))
    tau = [(7 * k + 3) % p for k in range(m.bit_length() - 1)]
    cv = O.CURVES[cid]
    cW, cE = cv.msm_known_dlog(W, K0, D), cv.msm_known_dlog(Er, K0, D)
    items = [(u, list(X), cW, cE, tau, pr.spartan_prove(gens, tau, SR.Transcript(q))) for q in range(kmax)]
    pr.close()
    nnz = len(A) + len(B) + len(Cm)
    unit = sum(1 for M in (A, B, Cm) for _, _, v in M if v % p in (1, p - 1))
    return dict(fid=fid, cid=cid, t=t, p=p, cons=cons, vars=nvars, io=io, m=m, nnz=nnz, f=(nnz - unit) / nnz,
                shape=gs, gens=gens, cv=cv, items=items)


class Call:
    """one vdfgpu_spartan_verify_batch call with its records encoded once"""

    def __init__(self, lib, _lib, sd, k):
        from vdf_b200 import spartan as SP
        from vdf_b200.encoding import fes_to_bytes
        self.rec = SP.spartan_records(sd["shape"], sd["cid"], sd["items"][:k])
        self.w = fes_to_bytes([3 * q + 1 for q in range(k)], sd["p"])
        self.k, self.ok = k, bytearray(k)
        self.args = [sd["shape"]._h, sd["gens"]._h, k] + [_lib.as_ptr(r) for r in self.rec] + \
                    [_lib.as_ptr(self.w), _lib.as_ptr(self.ok)]
        self.fn, self.check = lib.vdfgpu_spartan_verify_batch, _lib.check

    def __call__(self):
        self.check(self.fn(*self.args))
        return list(self.ok)


class Composed:
    """the path the call replaces: k x vdfgpu_r1cs_evaluate, one vdfgpu_ipa_verify_batch; every argument prepared"""

    def __init__(self, lib, _lib, sd, k):
        from oracle import pasta as O
        from tests import spartan_verify_ref as SVR
        from vdf_b200.encoding import fes_to_bytes
        p, cv, items = sd["p"], sd["cv"], sd["items"][:k]
        ell = sd["m"].bit_length() - 1
        self.evals = [(fes_to_bytes(pf.r_x, p) or bytes(32), fes_to_bytes(pf.r_y, p), bytearray(96))
                      for *_, pf in items]
        ops = [SVR.opening(cv, sd["fid"], it) for it in items]   # (Ls, Rs, rs, a_hat, comm_a, c, b_hat, u_scale)
        self.bufs = [b"".join(O.jac_to_bytes(cv, o[4]) for o in ops),
                     b"".join(O.jac_to_bytes(cv, L) for o in ops for L in o[0]) or bytes(96),
                     b"".join(O.jac_to_bytes(cv, R) for o in ops for R in o[1]) or bytes(96),
                     fes_to_bytes([r for o in ops for r in o[2]], p) or bytes(32)] + \
                    [fes_to_bytes([o[i] for o in ops], p) for i in (3, 5, 6, 7)] + \
                    [fes_to_bytes([3 * q + 1 for q in range(k)], p)]
        self.ok = bytearray(k)
        self.lib, self._lib, self.sd, self.k, self.ell = lib, _lib, sd, k, ell

    def __call__(self):
        lib, P = self.lib, self._lib.as_ptr
        for rx, ry, out in self.evals:
            self._lib.check(lib.vdfgpu_r1cs_evaluate(self.sd["shape"]._h, P(rx), P(ry), P(out)))
        self._lib.check(lib.vdfgpu_ipa_verify_batch(self.sd["gens"]._h, self.ell, self.k, *[P(b) for b in self.bufs],
                                                    P(self.ok)))
        return list(self.ok)


KERNELS = ("sparse_eval_batch_kernel", "EqHalfTablesBatchFn", "sc_column_sum_kernel")


def kernel_us(torch, fn, calls=3):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {"timer": "torch.profiler kernel records (CUPTI)", **{n: 0.0 for n in KERNELS}}
    for e in prof.key_averages():
        for name in KERNELS:
            if name in e.key:
                out[name] += e.device_time_total / calls
    return out


def host_ms(torch, call, calls=3):
    """per call: the start of its record_function range to the first runtime call that enqueues device work"""
    from torch.profiler import ProfilerActivity, profile, record_function
    call()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            with record_function("spartan_verify_batch_call"):
                call()
    evs = prof.events()
    cpu = torch.autograd.DeviceType.CPU
    ranges = sorted((e.time_range.start, e.time_range.end) for e in evs
                    if e.name == "spartan_verify_batch_call" and e.device_type == cpu)
    firsts, names = [], set()
    for t0, t1 in ranges:
        inside = sorted((e.time_range.start, e.name) for e in evs if e.name in DEVICE_WORK and t0 <= e.time_range.start <= t1)
        if inside:
            firsts.append((inside[0][0] - t0) / 1e3)
            names.add(inside[0][1])
    if not firsts:
        return {"method": "no runtime call recorded inside the call: not measured"}
    return {"method": "torch.profiler CPU timestamps, call start -> first " + "/".join(sorted(names)), **stats(firsts)}


def measure(lib, _lib, torch, sd, runs, warm):
    res = {"curve": "pallas" if sd["cid"] == 0 else "vesta", "t": sd["t"], "cons": sd["cons"], "vars": sd["vars"],
           "m": sd["m"], "ell_x": sd["m"].bit_length() - 1, "nnz": sd["nnz"], "f_non_unit": sd["f"], "by_k": []}
    mults_per_proof = sd["nnz"] * (1 + sd["f"]) + 4 * sd["cons"]
    res["mults_per_proof"] = mults_per_proof
    for k in (1, 8, 64):
        call, comp = Call(lib, _lib, sd, k), Composed(lib, _lib, sd, k)
        assert call() == [1] * k and comp() == [1] * k, "the proofs must verify on both paths"
        r = {"k": k}
        # the two paths alternated, so that both see the same state of the shared machine
        a, b = [], []
        for j in range(warm + runs):
            for fn, ts in ((call, a), (comp, b)):
                t0 = time.perf_counter()
                fn()
                if j >= warm:
                    ts.append((time.perf_counter() - t0) * 1e3)
        r["call_ms"], r["composed_ms"] = stats(a), stats(b)
        ku = kernel_us(torch, call)
        r["kernels_us"] = ku
        r["mults"] = k * mults_per_proof
        if ku["sparse_eval_batch_kernel"] > 0:
            rate = r["mults"] / (ku["sparse_eval_batch_kernel"] * 1e-6)
            r["mul_per_s"] = rate
            r["fraction_of_multiplier"] = rate / MUL_RATE
        if k == 64:
            r["host_ms"] = host_ms(torch, call)
        print(json.dumps({"curve": res["curve"], "t": sd["t"], **r}), flush=True)
        res["by_k"].append(r)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r4_spartan_verify.json"))
    ap.add_argument("--runs", type=int, default=7)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--ts", default="10,1024,16384", help="primary step rounds")
    args = ap.parse_args()
    import torch
    from profile_verify import device_info
    from vdf_b200 import _lib
    if not torch.cuda.is_available():
        raise SystemExit("profile_spartan_verify: no CUDA device (the measurement has no CPU fallback)")
    lib = _lib.load()
    _lib.check(lib.vdfgpu_init(0))
    res = {"device": device_info(), "configs": []}
    sides = [(1, 0, int(t), 9800, 42) for t in args.ts.split(",")] + [(0, 1, 0, 10300, 7)]
    for fid, cid, t, aug, seed in sides:
        sd = side(fid, cid, t, aug, seed, 64)
        res["configs"].append(measure(lib, _lib, torch, sd, args.runs, args.warm))
        sd["gens"].close()
        sd["shape"].close()
    res["note"] = ("augmented blocks SYNTHETIC; composed_ms leaves out the host sum-check checks and the derivation of "
                   "c, b_hat and comm_E + rho comm_W, which favours it; weights 3q + 1")
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
