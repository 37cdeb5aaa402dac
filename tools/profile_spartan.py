#!/usr/bin/env python
"""RelaxedR1CSSNARK::prove of a resident running instance in one call (vdfgpu_running_spartan_prove) at the step shapes
of bench.py: primary (Pallas, t = 10, 1024, 16384, SYNTHETIC 9.8k-constraint augmented block) and secondary (Vesta,
SYNTHETIC 10.3k-constraint augmented circuit, no step rounds).  The running instance is satisfied and relaxed: u != 1
and E = Az.Bz - u.Cz (dense).  The IPA set: a table-layout progression of m + 1 points.  Per shape:
  prove_ms          wall time of the call with a sha256 transcript in Python callbacks; median and min after warm-up
  callbacks_ms      the part of it spent inside the Python callbacks (timed in them)
  phases_ms         CUDA events recorded on the call's stream from inside the callbacks at the phase boundaries, so
                    each phase includes its own callbacks: outer (snapshot, outer sum-check, its claims), bind + scatter
                    (to the first inner round's callback: inner tables and the first inner round), inner (the other
                    inner rounds and the evaluation claims), ipa (joint claim and the inner-product argument)
  block_path_ms     the same proof by the entry points it replaces: vdfgpu_running_get, then host vectors through
                    vdfgpu_multiply_vec, vdfgpu_eq_evals, vdfgpu_sumcheck_cubic / _quad, vdfgpu_poly_evaluate,
                    vdfgpu_r1cs_bind_rows, vdfgpu_inner_product, vdfgpu_vec_lincomb and vdfgpu_ipa_prove, with the
                    padding and u Cz + E done in Python integers in between
  evaluate_ms       vdfgpu_r1cs_evaluate alone
And both curves proved concurrently from two threads on their own streams (t = 16384 primary with the secondary), wall
time of the pair.  Writes one JSON line (default profiles/r3_spartan.json) with the device name, power limit and max SM
clock read in the same run."""
import argparse
import hashlib
import json
import statistics
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

K0, D = 1234567, 89


def stats(ts):
    return {"median": statistics.median(ts), "min": min(ts), "runs": len(ts)}


class Sha:
    """a transcript: sha256 of everything handed over, timed; optional per-phase CUDA events on stream s"""

    def __init__(self, p, torch=None, s=None):
        self.p, self.torch, self.s = p, torch, s
        self.cb = 0.0
        self.events = {}
        self.stage = 0

    def _h(self, *xs):
        return int.from_bytes(hashlib.sha256(repr(xs).encode()).digest(), "little") % self.p or 1

    def _mark(self, name):
        if self.s is not None and name not in self.events:
            e = self.torch.cuda.Event(enable_timing=True)
            e.record(self.s)
            self.events[name] = e

    def sumcheck_round(self, rnd, evals):
        t0 = time.perf_counter()
        if self.stage == 1 and rnd == 0:
            self._mark("inner0")
        r = self._h(rnd, evals)
        self.cb += time.perf_counter() - t0
        return r

    def claims(self, stage, values):
        t0 = time.perf_counter()
        self._mark(("outer", "inner", "ipa")[stage])
        self.stage = stage + 1
        out = [self._h(stage, values, k) for k in range((3, 1, 1)[stage])]
        self.cb += time.perf_counter() - t0
        return out

    def ipa_round(self, rnd, L, R):
        t0 = time.perf_counter()
        r = self._h(rnd, L, R)
        self.cb += time.perf_counter() - t0
        return r


def side(fid, cid, t, aug, seed):
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
    return dict(fid=fid, cid=cid, t=t, p=p, cons=cons, vars=nvars, io=io, m=m, shape=gs, gens=gens, prover=pr, tau=tau)


def measure(lib, _lib, torch, sd, runs, warm, block):
    s = torch.cuda.Stream()
    _lib.check(lib.vdfgpu_set_stream(s.cuda_stream))
    try:
        return measure_on_stream(lib, _lib, torch, sd, s, runs, warm, block)
    finally:
        torch.cuda.synchronize()
        _lib.check(lib.vdfgpu_set_stream(None))


def measure_on_stream(lib, _lib, torch, sd, s, runs, warm, block):
    p, pr, gens, tau = sd["p"], sd["prover"], sd["gens"], sd["tau"]
    walls, cbs, phases = [], [], {k: [] for k in ("outer", "bind_scatter", "inner", "ipa")}
    pf = None
    for k in range(warm + runs):
        tr = Sha(p, torch, s)
        torch.cuda.synchronize()
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record(s)
        t0 = time.perf_counter()
        pf = pr.spartan_prove(gens, tau, tr)
        wall = (time.perf_counter() - t0) * 1e3
        end.record(s)
        end.synchronize()
        if k >= warm:
            walls.append(wall)
            cbs.append(tr.cb * 1e3)
            ev = tr.events
            phases["outer"].append(start.elapsed_time(ev["outer"]))
            phases["bind_scatter"].append(ev["outer"].elapsed_time(ev["inner0"]))
            phases["inner"].append(ev["inner0"].elapsed_time(ev["ipa"]))
            phases["ipa"].append(ev["ipa"].elapsed_time(end))
    out = {"curve": "pallas" if sd["cid"] == 0 else "vesta", "t": sd["t"], "cons": sd["cons"], "vars": sd["vars"],
           "m": sd["m"], "ell_x": sd["m"].bit_length() - 1, "prove_ms": stats(walls), "callbacks_ms": stats(cbs),
           "phases_ms": {k: statistics.median(v) for k, v in phases.items()}}
    ts = []
    for k in range(warm + runs):
        t0 = time.perf_counter()
        sd["shape"].evaluate(pf.r_x, pf.r_y)
        if k >= warm:
            ts.append((time.perf_counter() - t0) * 1e3)
    out["evaluate_ms"] = stats(ts)
    if block:
        ts = []
        for k in range(1 + max(2, runs // 2)):
            t0 = time.perf_counter()
            block_path(lib, _lib, sd)
            if k:
                ts.append((time.perf_counter() - t0) * 1e3)
        out["block_path_ms"] = stats(ts)
    return out


def block_path(lib, _lib, sd):
    """the proof from host vectors; the transcript is the same sha256 stand-in"""
    from vdf_b200 import spartan as SP
    fid, p, gs, pr, gens, tau = sd["fid"], sd["p"], sd["shape"], sd["prover"], sd["gens"], sd["tau"]
    cons, nvars, io, m = sd["cons"], sd["vars"], sd["io"], sd["m"]
    tr = Sha(p)
    W, Ev, u, X = pr.get_running()                       # vdfgpu_running_get
    Az, Bz, Cz = gs.multiply_vec(list(W) + [u] + list(X))
    pad = lambda v, n: list(v) + [0] * (n - len(v))      # noqa: E731
    D = [(u * c + e) % p for c, e in zip(Cz, Ev)]
    _, rx, fin = SP.sumcheck(fid, [SP.eq_evals(fid, tau), pad(Az, m), pad(Bz, m), pad(D, m)], tr.sumcheck_round)
    claim_Cz, eval_E = SP.poly_evaluate(fid, pad(Cz, m), rx), SP.poly_evaluate(fid, pad(Ev, m), rx)
    r_abc = tr.claims(0, (fin[1], fin[2], claim_Cz, eval_E))
    eq_rx = SP.eq_evals(fid, rx)
    Mc = gs.bind_rows(eq_rx[:cons], r_abc)
    Mp = Mc[:nvars] + [0] * (m - nvars) + Mc[nvars:] + [0] * (m - 1 - io)
    zp = list(W) + [0] * (m - nvars) + [u] + list(X) + [0] * (m - 1 - io)
    _, ry, _ = SP.sumcheck(fid, [Mp, zp], tr.sumcheck_round)
    eq_ry = SP.eq_evals(fid, ry[1:])
    eval_W = SP.poly_evaluate(fid, pad(W, m), ry[1:])
    T = (SP.inner_product(fid, pad(Ev, m), eq_ry) + SP.inner_product(fid, pad(W, m), eq_rx)) % p
    (rho,) = tr.claims(1, (eval_W, T))
    a = SP.vec_lincomb(fid, pad(Ev, m), pad(W, m), 1, rho)
    b = SP.vec_lincomb(fid, eq_rx, eq_ry, 1, rho)
    c = (eval_E + rho * T + rho * rho * eval_W) % p
    (u_scale,) = tr.claims(2, (c,))
    SP.ipa_prove(gens, a, b, u_scale, tr.ipa_round)


def concurrent(lib, _lib, torch, sides, runs, warm):
    """both sides proved at once from two threads, each on its own stream; wall time of the pair"""
    streams = [torch.cuda.Stream() for _ in sides]
    ts = []
    for k in range(warm + runs):
        torch.cuda.synchronize()
        errs = []

        def run(sd, s):
            try:
                _lib.check(lib.vdfgpu_set_stream(s.cuda_stream))
                sd["prover"].spartan_prove(sd["gens"], sd["tau"], Sha(sd["p"]))
                _lib.check(lib.vdfgpu_set_stream(None))
            except Exception as e:   # noqa: BLE001
                errs.append(e)
        th = [threading.Thread(target=run, args=(sd, s)) for sd, s in zip(sides, streams)]
        t0 = time.perf_counter()
        for t in th:
            t.start()
        for t in th:
            t.join()
        if errs:
            raise errs[0]
        if k >= warm:
            ts.append((time.perf_counter() - t0) * 1e3)
    return stats(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_spartan.json"))
    ap.add_argument("--runs", type=int, default=7)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--ts", default="10,1024,16384", help="primary step rounds")
    args = ap.parse_args()
    import torch
    from profile_verify import device_info
    from vdf_b200 import _lib
    if not torch.cuda.is_available():
        raise SystemExit("profile_spartan: no CUDA device (the measurement has no CPU fallback)")
    lib = _lib.load()
    _lib.check(lib.vdfgpu_init(0))
    res = {"device": device_info(), "configs": []}
    sec = side(0, 1, 0, 10300, 7)
    pri = None
    for t in [int(x) for x in args.ts.split(",")]:
        pri = side(1, 0, t, 9800, 42)
        r = measure(lib, _lib, torch, pri, args.runs, args.warm, block=True)
        print(json.dumps(r), flush=True)
        res["configs"].append(r)
    r = measure(lib, _lib, torch, sec, args.runs, args.warm, block=True)
    print(json.dumps(r), flush=True)
    res["configs"].append(r)
    res["concurrent_ms"] = {"primary_t": pri["t"], "pair": concurrent(lib, _lib, torch, [pri, sec], args.runs,
                                                                         args.warm)}
    res["note"] = ("callbacks: a sha256 stand-in for nova's Poseidon transcript in Python; augmented blocks SYNTHETIC; "
                   "block_path does the padding and u Cz + E in Python integers")
    print(json.dumps(res["concurrent_ms"]), flush=True)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
