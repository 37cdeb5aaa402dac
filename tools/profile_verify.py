#!/usr/bin/env python
"""The GPU side of RecursiveSNARK::verify (src/nova/proof.rs:382) at Nova sizes, and the row-check kernel alone.

Per t in (10, 100, 1000, 1024, 4096, 16384), with the shapes of bench.py's nova_step_measurements (synthetic step
instance + 9 800-constraint block on the primary curve, 10 300-constraint block on the secondary):
  verify_ms         primary is_sat_relaxed + secondary is_sat_relaxed + secondary is_sat from HOST vectors, each call
                    ending in a synchronise: back to back, and the three from three host threads
  running_check_ms  vdfgpu_running_check on the resident primary and secondary running instances
  cpu_port_ms       the same three checks' mat-vecs and MSMs with oracle/cpu_ref.c on all host cores ("port"; it
                    leaves out the O(cons) row products, which favours the CPU)
The row-check kernel alone: vdfgpu_r1cs_is_sat_relaxed_dev on bench.py's 2^21-constraint extra.r1cs_hbm shape, "unit"
and "random_B" coefficient mixes, CUDA events over many launches (inputs about 0.4 GB, larger than L2), against the
device-to-device copy bandwidth measured in the same run.
Writes one JSON line (default profiles/r3_verify.json) with the device name and power limit read in the same run."""
import argparse
import ctypes
import json
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


def device_info():
    """nvidia-smi, read-only: what the numbers were measured on."""
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [s.strip() for s in out.split(",")]))
    except Exception as e:   # noqa: BLE001
        return {"error": repr(e)}


def wall_ms(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return {"median": statistics.median(ts), "min": min(ts), "reps": reps}


def in_threads(lib, fns, streams):
    """Run each callable on its own host thread with its own CUDA stream (vdfgpu_set_stream is per thread; ctypes
    releases the GIL in the library call); returns when all have ended."""
    def run(f, s):
        lib.vdfgpu_set_stream(s)
        f()
    ths = [threading.Thread(target=run, args=(f, s)) for f, s in zip(fns, streams)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()


def verify_measurements(lib, _lib, torch, ts, reps, cpu):
    from oracle import cpu_ref as C, pasta as O
    from vdf_b200 import encoding as E, msm as G, nova as N, synthetic as S
    K0, D = 11, 7
    u_relaxed = 0x1234567890ABCDEF1234567890ABCDEF

    def side(fid, cid, t, aug, seed):
        """A satisfied relaxed running instance with u != 1 and a dense error vector E = Az.Bz - u.Cz (a fold of the
        synthetic witness with itself would leave E = 0, whose commitment is cheaper than a real one), and the fresh
        instance (u = 1, E = 0) for the strict check."""
        cons, nvars, io, A, B, Cm, W, X = S.step_instance(fid, t, aug, seed=seed)
        gs = N.R1CSShape(fid, cons, nvars, io, A, B, Cm)
        gens = G.Generators.progression(cid, K0, D, max(cons, nvars), table=True)
        m = E.MODULUS[fid]
        u = u_relaxed
        Az, Bz, Cz = gs.multiply_vec(list(W) + [u] + list(X))
        Er = [(a * b - u * c) % m for a, b, c in zip(Az, Bz, Cz)]
        U = N.RelaxedR1CSInstance(gens.commit(W), gens.commit(Er), list(X), u)
        pr = N.RunningProver(gs, gens)
        pr.set_running(W, Er, U)
        base = E.CURVE_BASE[cid]
        jac = lambda p: E.fe_to_bytes(p[0], base) + E.fe_to_bytes(p[1], base) + E.fe_to_bytes(1, base)  # noqa: E731
        d = dict(fid=fid, cid=cid, shape=gs, gens=gens, prover=pr, cons=cons, nvars=nvars, io=io, coo=(A, B, Cm),
                 W=E.fes_to_bytes(W, m), E=E.fes_to_bytes(Er, m), u=E.fe_to_bytes(u, m), X=E.fes_to_bytes(X, m),
                 cW=jac(U.comm_W), cE=jac(U.comm_E), W1=E.fes_to_bytes(W, m), X1=E.fes_to_bytes(X, m),
                 cW1=jac(U.comm_W), m=m, E_nonzero=sum(1 for e in Er if e))
        return d

    def call(s, strict=False):
        rep = (ctypes.c_uint64 * 4)()
        if strict:
            _lib.check(lib.vdfgpu_r1cs_is_sat_relaxed(s["shape"]._h, s["gens"]._h, s["W1"], None, None, s["X1"],
                                                      s["cW1"], None, rep))
        else:
            _lib.check(lib.vdfgpu_r1cs_is_sat_relaxed(s["shape"]._h, s["gens"]._h, s["W"], s["E"], s["u"], s["X"],
                                                      s["cW"], s["cE"], rep))
        return list(rep)

    def running(s):
        rep = (ctypes.c_uint64 * 4)()
        _lib.check(lib.vdfgpu_running_check(s["prover"]._h, s["cW"], s["cE"], rep))
        return list(rep)

    sec = side(E.FP, 1, 0, 10300, 7)
    keep = [torch.cuda.Stream() for _ in range(3)]
    streams = [s.cuda_stream for s in keep]
    out = {}
    for t in ts:
        pri = side(E.FQ, 0, t, 9800, 42)
        reports = [call(pri), call(sec), call(sec, strict=True), running(pri), running(sec)]
        for rep, s in zip(reports, (pri, sec, sec, pri, sec)):
            if rep[:2] != [0, s["cons"]] or 0 in rep[2:]:
                raise RuntimeError(f"t = {t}: a satisfied instance was reported {rep}")
        entry = {"primary_cons": pri["cons"], "primary_vars": pri["nvars"], "secondary_cons": sec["cons"],
                 "secondary_vars": sec["nvars"], "primary_E_nonzero": pri["E_nonzero"],
                 "secondary_E_nonzero": sec["E_nonzero"], "reports_satisfied": True}
        entry["verify_ms"] = wall_ms(lambda: (call(pri), call(sec), call(sec, strict=True)), reps)
        entry["verify_ms_3_threads"] = wall_ms(lambda: in_threads(lib, [lambda: call(pri), lambda: call(sec),
                                                                        lambda: call(sec, strict=True)], streams), reps)
        entry["running_check_ms"] = wall_ms(lambda: (running(pri), running(sec)), reps)
        entry["primary_is_sat_relaxed_ms"] = wall_ms(lambda: call(pri), reps)
        entry["primary_rows_only_ms"] = wall_ms(
            lambda: _lib.check(lib.vdfgpu_r1cs_is_sat_relaxed(pri["shape"]._h, None, pri["W"], pri["E"], pri["u"], pri["X"],
                                                              None, None, (ctypes.c_uint64 * 4)())), reps)
        if cpu:
            entry["cpu_port_ms"] = cpu_port(C, O, lib, _lib, pri, sec)
        out[str(t)] = entry
        pri["prover"].close(); pri["gens"].close(); pri["shape"].close()
    sec["prover"].close(); sec["gens"].close(); sec["shape"].close()
    return out


def cpu_port(C, O, lib, _lib, pri, sec):
    """Mat-vecs and MSMs of the three checks with the C port on all host cores (best of two)."""
    cores = C.ncores()
    parts = []
    for s, strict in ((pri, False), (sec, False), (sec, True)):
        ngen = max(s["cons"], s["nvars"])
        pts = bytearray(72 * ngen)
        _lib.check(lib.vdfgpu_gens_export(s["gens"]._h, 0, ngen, _lib.as_ptr(pts)))
        coo = O.shape_to_coo_bytes(O.R1CSShape(s["m"], s["cons"], s["nvars"], s["io"], *s["coo"]))
        parts.append((s, strict, bytes(pts), coo))
    best = None
    for _ in range(2):
        t0 = time.perf_counter()
        for s, strict, pts, coo in parts:
            fid = s["fid"]
            if strict:
                C.multiply_vec(fid, s["cons"], s["nvars"], s["io"], coo, s["W1"], O.fe_to_bytes(1, s["m"]), s["X1"])
                C.msm(s["cid"], pts[:72 * s["nvars"]], s["W1"], True, cores)
            else:
                C.multiply_vec(fid, s["cons"], s["nvars"], s["io"], coo, s["W"], s["u"], s["X"])
                C.msm(s["cid"], pts[:72 * s["nvars"]], s["W"], True, cores)
                C.msm(s["cid"], pts[:72 * s["cons"]], s["E"], True, cores)
        dt = (time.perf_counter() - t0) * 1e3
        best = dt if best is None else min(best, dt)
    return {"ms": best, "cores": cores, "kind": "port",
            "note": "mat-vecs and MSMs only; the O(cons) row products Az*Bz - u*Cz - E are not timed (favours the CPU)"}


def copy_bandwidth(torch, gib=2):
    """Device-to-device copy of a `gib` GiB buffer: 2 x bytes per copy, CUDA events, best of 10."""
    n = gib << 30
    a = torch.empty(n, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    best = None
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        torch.cuda.synchronize()
        s = e0.elapsed_time(e1) * 1e-3
        best = s if best is None else min(best, s)
    del a, b
    return 2 * n / best / 1e9


def row_kernel_measurements(lib, _lib, torch, hbm_gbs, log2rows=21, launches=50):
    """vdfgpu_r1cs_is_sat_relaxed_dev on bench.py's extra.r1cs_hbm shape.  W = X = 0 and E = 0 make every row hold
    (the case of real use) while the kernel reads exactly the same bytes; the random-input case (every row violated:
    one atomic pair per warp) is timed beside it."""
    import numpy as np
    import bench
    from vdf_b200.encoding import Q, fe_to_bytes
    cons = vars_ = 1 << log2rows
    io = 2
    r = np.arange(cons, dtype=np.uint64)
    one, neg1, rnd = fe_to_bytes(1, Q), fe_to_bytes(Q - 1, Q), fe_to_bytes(0x1234567890ABCDEF1234567890ABCDEF, Q)
    a_rows, a_cols = r, r
    b_rows, b_cols = r, np.ascontiguousarray((r * 7 + 3) % vars_)
    c_rows = np.concatenate([r, r])
    c_cols = np.ascontiguousarray(np.concatenate([(r + 1) % vars_, (r * 5) % vars_]))
    a_vals = np.frombuffer(one * cons, dtype=np.uint8)
    c_vals = np.frombuffer(one * cons + neg1 * cons, dtype=np.uint8)
    nnz = 4 * cons
    alg = 36 * nnz + 4 * (3 * cons + 1) + 32 * (vars_ + 1 + io) + 32 * cons
    zeros = {k: torch.zeros((n, 4), dtype=torch.int64, device="cuda") for k, n in (("W", vars_), ("E", cons), ("uX", 1 + io))}
    zeros["uX"][0] = torch.tensor(np.frombuffer(one, dtype=np.int64).copy())
    rand = {"W": bench.rand_fe_dev(torch, vars_), "E": bench.rand_fe_dev(torch, cons), "uX": bench.rand_fe_dev(torch, 1 + io)}
    counts = torch.zeros(2, dtype=torch.int64, device="cuda")
    res = {"shape": {"cons": cons, "vars": vars_, "nnz": nnz}, "algorithmic_bytes": alg,
           "bytes_formula": "36 nnz + 4 (3 cons + 1) + 32 (vars + 1 + io) + 32 cons", "launches_timed": launches}
    for mix, bval in (("unit", one), ("random_B", rnd)):
        b_vals = np.frombuffer(bval * cons, dtype=np.uint8)
        h = ctypes.c_void_p()
        _lib.check(lib.vdfgpu_r1cs_create(1, cons, vars_, io,
                                          a_rows.ctypes.data, a_cols.ctypes.data, a_vals.ctypes.data, cons,
                                          b_rows.ctypes.data, b_cols.ctypes.data, b_vals.ctypes.data, cons,
                                          c_rows.ctypes.data, c_cols.ctypes.data, c_vals.ctypes.data, 2 * cons,
                                          ctypes.byref(h)))
        out = {}
        for case, v in (("rows_hold", zeros), ("every_row_violated", rand)):
            fn = lambda: _lib.check(lib.vdfgpu_r1cs_is_sat_relaxed_dev(h, v["W"].data_ptr(), v["E"].data_ptr(),  # noqa: E731
                                                                      v["uX"].data_ptr(), counts.data_ptr()))
            s = bench.cuda_timed(torch, fn, reps=launches, warm=3)
            got = counts.cpu().tolist()
            out[case] = {"ms": s * 1e3, "achieved_gbs": alg / s / 1e9, "frac_of_measured_hbm": alg / s / 1e9 / hbm_gbs,
                         "violating_rows": got[0], "first_violating_row": got[1]}
        out["coefficients"] = "A = +1, B = full-size random, C = +1 / -1" if mix == "random_B" else "all +1 / -1 (step-circuit mix)"
        res[mix] = out
        _lib.check(lib.vdfgpu_r1cs_destroy(h))
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_verify.json"))
    ap.add_argument("--ts", default="10,100,1000,1024,4096,16384")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--no-cpu", action="store_true", help="skip the C-port timing")
    a = ap.parse_args()
    import torch
    from vdf_b200 import _lib
    if not torch.cuda.is_available():
        raise SystemExit("profile_verify: no CUDA device (the measurement has no CPU fallback)")
    lib = _lib.load()
    _lib.check(lib.vdfgpu_init(0))
    # the library enqueues on the calling thread's stream: make it torch's current one, or the CUDA events of
    # bench.cuda_timed would time an empty stream
    st = torch.cuda.Stream()
    torch.cuda.set_stream(st)
    _lib.check(lib.vdfgpu_set_stream(st.cuda_stream))
    res = {"device": device_info()}
    hbm = copy_bandwidth(torch)
    res["hbm_copy_gbs"] = hbm
    import bench
    res["hbm_peak_bench"] = bench.hbm_peak()
    res["row_kernel"] = row_kernel_measurements(lib, _lib, torch, hbm)
    res["verify"] = verify_measurements(lib, _lib, torch, [int(x) for x in a.ts.split(",")], a.reps, not a.no_cpu)
    res["note"] = ("verify_ms: primary is_sat_relaxed + secondary is_sat_relaxed + secondary is_sat from host vectors "
                   "(each with its commitments, each ending in a synchronise); augmented blocks SYNTHETIC; Poseidon hash "
                   "checks not included. cpu_port_ms: mat-vecs and MSMs only, on all host cores")
    res["device_after"] = device_info()
    line = json.dumps(res)
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
