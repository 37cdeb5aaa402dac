#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path: Pallas MSM Gpoints/s (BASELINE.json metric), with the
fold-step, batched-verify, size-sweep, strong-scaling and drop-in measurements as extra keys on the same JSON line.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--log2n L] [--dump-outputs DIR]

One "step" = one commitment MSM over n = 2^L synthetic scalars against a device-resident generator set
(P_i = (k0 + i d) G, generated on the device; generators are fixed for the life of PublicParams in the
reference, src/nova/proof.rs:232-237).  N > 1 (torchrun, one rank per GPU): each rank owns a contiguous point
range of n points (weak scaling), emits one un-normalised partial point, and the 96-byte partials are all-gathered
(NCCL) and summed + normalised once on every rank -- SURVEY.md section 8(e).

`value`  : device-timed (CUDA events), scalars already in HBM, K independent commitments with `plan.inflight`
           of them in flight (alternating streams: the latency-bound stages of one MSM run under the multiply-bound
           kernels of the next); `serial` on the same line is the one-at-a-time figure.
`e2e`    : the same step through the reference-facing C ABI with HOST scalars (H2D of n*32 B and D2H of the 96-byte
           commitment inside the timed region), three ways: pipelined from pinned memory (value), one synchronous
           call at a time from pinned memory, and from pageable memory (what a Rust Vec is).
`--impl reference`: the CPU restatement of the reference's pasta-msm Pippenger (oracle/cpu_ref.c, all host cores)
           on the same workload; the Rust crates cannot be built here.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "Pallas MSM Gpoints/s"
print_json = print
K0, D = 0x1234567, 0x89ABCDEF01
MUL32_PER_FIELD_MUL = 136        # SURVEY.md 8(d): generic CIOS, n = 8 limbs: 2n^2 + n
FIELD_MUL_PER_MADD = 10          # XYZZ mixed addition 8M + 2S
Q_ORDER = 0x40000000000000000000000000000000224698FC0994A8DD8C46EB2100000001   # Pallas group order


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2n", type=int, default=22, help="points per GPU = 2^log2n")
    ap.add_argument("--plain", action="store_true", help="plain generator layout instead of the table")
    ap.add_argument("--inflight", type=int, default=4, choices=[1, 2, 3, 4], help="independent commitments in flight in the device-timed region and in the pipelined e2e")
    ap.add_argument("--no-extra", action="store_true", help="skip every side measurement")
    ap.add_argument("--no-sweep", action="store_true", help="skip the 2^20..2^26 size sweep / strong-scaling leg")
    ap.add_argument("--cpu-budget-s", type=float, default=150.0, help="wall-time budget of the CPU reference arm")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy "
                    "(float64), to compare two builds output for output")
    return ap.parse_args()


def dump_outputs(out_dir: str, points96: dict) -> None:
    """Each 96-byte point (X, Y, Z; four little-endian u64 limbs per coordinate, Montgomery form, include/vdfgpu.h) as
    DIR/<name>.npy: a (3, 8) float64 array of its 32-bit limbs, which float64 holds exactly."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, b in points96.items():
        limbs = np.frombuffer(bytes(b), dtype="<u4").reshape(3, 8)
        np.save(os.path.join(out_dir, f"{name}.npy"), limbs.astype(np.float64))


def workload_config(log2n: int, world: int):
    """`config` shared verbatim by both arms (the driver compares it)."""
    return {"workload": f"Pallas MSM (BASELINE config 2/5), n = 2^{log2n} points per GPU, uniform 254-bit scalars, "
                        f"known-dlog points (k0 + i d) G",
            "points_per_gpu": 1 << log2n, "points_total": world * (1 << log2n),
            "l2": "inputs larger than L2 (scalars 32 B/pt + point table 64 B/pt/level >> 126 MB); no flush needed",
            "parallelism": (f"point-range shards x{world}, all-gather of 96-byte un-normalised partials, one warp sums and "
                            f"normalises") if world > 1 else "single GPU"}


# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def visible_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except (ValueError, IndexError):
            return local_rank
    return local_rank


# ---------------------------------------------------------------------------------------------------
def cpu_msm_timed(points72: bytes, scalars: bytes, max_reps: int = 2):
    """oracle/cpu_ref.c MSM (restatement of pasta-msm's CPU Pippenger) on all host cores; best of max_reps."""
    from oracle import cpu_ref as C
    cores = C.ncores()
    n = len(scalars) // 32
    C.msm(0, points72[:72 * 4096], scalars[:32 * 4096], True, cores)  # warm-up (thread pool, page faults)
    best, out = None, None
    for _ in range(max_reps):
        t0 = time.perf_counter()
        out = C.msm(0, points72, scalars, True, cores)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return {"value": n / best / 1e9, "unit": "Gpoints/s", "cores": cores, "kind": "port",
            "sample": f"Pallas MSM over the FULL workload n=2^{n.bit_length() - 1} (same points and scalars as the GPU arm), "
                      f"best of {max_reps} runs, {best * 1e3:.0f} ms each (oracle/cpu_ref.c: C restatement of pasta-msm's CPU "
                      f"Pippenger with MULX/ADX field arithmetic and a persistent thread pool; the Rust crates cannot be built here)"}, out


def run_reference(args):
    """CPU arm: the reference algorithm on the host cores; rank 0 only.  Same config as the GPU arm: every step is one
    MSM over n = 2^log2n points unless the wall-time budget forces a smaller per-step sample (stated in the line)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np
    from oracle import cpu_ref as C
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    cores = C.ncores()
    n_full = 1 << args.log2n
    rs = np.random.RandomState(42)

    def make(n):
        raw = rs.randint(0, 1 << 32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
        raw[:, 7] &= 0x3FFFFFFF
        return C.progression(0, K0, D, n, cores), raw.tobytes()

    # size the per-step sample from a probe so that (steps + warmup) steps fit the budget
    probe_n = min(n_full, 1 << 18)
    pts, scal = make(probe_n)
    C.msm(0, pts, scal, True, cores)
    t0 = time.perf_counter()
    C.msm(0, pts, scal, True, cores)
    per_point = (time.perf_counter() - t0) / probe_n
    total_steps = args.steps + max(1, args.warmup)
    n = n_full
    while n > probe_n and per_point * n * total_steps > args.cpu_budget_s:
        n >>= 1
    if n != probe_n:
        pts, scal = make(n)
    for _ in range(max(1, args.warmup)):
        C.msm(0, pts, scal, True, cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = C.msm(0, pts, scal, True, cores)
    dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"commitment": out})
    v = n / dt / 1e9
    same = n == n_full
    sample = (f"each step = one Pallas MSM over {'the full' if same else 'a bounded sample of'} n=2^{n.bit_length() - 1} points "
              f"{'(same per-GPU workload as the GPU arm)' if same else f'of the 2^{args.log2n}-point workload (wall-time budget {args.cpu_budget_s:.0f} s)'}; "
              f"oracle/cpu_ref.c, C restatement of pasta-msm's CPU Pippenger (MULX/ADX field arithmetic, persistent "
              f"thread pool), {cores} threads; Gpoints/s of one host, not scaled by the GPU count")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "Gpoints/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs (255-bit Montgomery, exact)", "data": "synthetic",
            "config": workload_config(args.log2n, world),
            "cpu_baseline": {"value": v, "unit": "Gpoints/s", "cores": cores, "kind": "port", "sample": sample},
            "sample_points_per_step": n, "same_points_per_step_as_gpu_arm": same,
            "e2e": {"value": v, "unit": "Gpoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print_json(json.dumps(line))


# ---------------------------------------------------------------------------------------------------
def hbm_peak():
    mp = ROOT / "MEASURED_PEAKS.json"
    if mp.exists():
        return float(json.loads(mp.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 7700.0, "fallback (B200_PROFILING.md nominal)"


def hbm_view(n, stage_s, traffic):
    """The same stage against the HBM roofline (the contract's other bound): compulsory bytes are one 32-byte scalar
    and one 64-byte point per MSM point, so this stage sits orders of magnitude under the HBM limit by algorithmic
    bytes; `traffic_gbs` is what ncu saw it really move."""
    peak, src = hbm_peak()
    alg = float(n) * 96
    out = {"bound": "hbm", "algorithmic_bytes": alg, "achieved": alg / stage_s / 1e9, "peak": peak, "unit": "GB/s",
           "frac": alg / stage_s / 1e9 / peak, "peak_source": src}
    if traffic:
        out["traffic_gbs"] = traffic / stage_s / 1e9
        out["traffic_frac_of_peak"] = traffic / stage_s / 1e9 / peak
    return out


def cuda_timed(torch, fn, reps=5, warm=2):
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e-3


def rand_fe_dev(torch, n, gen=None):
    """n uniform 254-bit values as (n, 4) int64 on the device: valid Montgomery-form field elements."""
    t = torch.randint(-(1 << 63), (1 << 63) - 1, (n, 4), dtype=torch.int64, device="cuda", generator=gen)
    t[:, 3] &= (1 << 62) - 1
    return t


def r1cs_hbm_measurements(lib, _lib, torch, log2rows: int = 21):
    """HBM-roofline leg for the R1CS kernels (SURVEY 8d): cross-term, multiply_vec and fold on an ENLARGED
    synthetic shape (2^21 constraints, 4 non-zeros per constraint row triple: the step circuit's density) so
    the data (about 0.5 GB) do not sit in L2.  Device-resident operands, CUDA events.  Two coefficient mixes:
    "unit" = every coefficient +1 / -1 (the MinRoot step circuit, src/nova/proof.rs:176-227: the add/sub fast path)
    and "random_B" = the B matrix holds full-size random coefficients (one real multiplication per B entry)."""
    import numpy as np
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
    W1, W2, E1 = rand_fe_dev(torch, vars_), rand_fe_dev(torch, vars_), rand_fe_dev(torch, cons)
    uX1, uX2, rr = rand_fe_dev(torch, 1 + io), rand_fe_dev(torch, 1 + io), rand_fe_dev(torch, 1)
    T = torch.zeros((cons, 4), dtype=torch.int64, device="cuda")
    ABC = torch.zeros((3 * cons, 4), dtype=torch.int64, device="cuda")
    peak, src = hbm_peak()
    res = {"shape": {"cons": cons, "vars": vars_, "nnz": nnz}, "hbm_peak_gbs": peak, "hbm_peak_source": src}
    b_ct = 36 * nnz + 4 * (3 * cons + 1) + 2 * 32 * (vars_ + 1 + io) + 32 * cons
    b_mv = 36 * nnz + 4 * (3 * cons + 1) + 32 * (vars_ + 1 + io) + 3 * 32 * cons
    b_fd = 96 * (vars_ + cons)
    # scaled row table (read cons, write 3 cons) + per entry: its stacked row (u32), the value, one gathered table element
    b_br = 32 * 4 * cons + (4 + 32 + 32) * nnz + 4 * (vars_ + 1 + io + 1) + 32 * (vars_ + 1 + io)
    rr3 = rand_fe_dev(torch, 3)
    Mt = torch.zeros((vars_ + 1 + io, 4), dtype=torch.int64, device="cuda")
    for mix, bval in (("random_B", rnd), ("unit", one)):
        b_vals = np.frombuffer(bval * cons, dtype=np.uint8)
        h = ctypes.c_void_p()
        _lib.check(lib.vdfgpu_r1cs_create(1, cons, vars_, io,
                                          a_rows.ctypes.data, a_cols.ctypes.data, a_vals.ctypes.data, cons,
                                          b_rows.ctypes.data, b_cols.ctypes.data, b_vals.ctypes.data, cons,
                                          c_rows.ctypes.data, c_cols.ctypes.data, c_vals.ctypes.data, 2 * cons,
                                          ctypes.byref(h)))
        t_ct = cuda_timed(torch, lambda: _lib.check(lib.vdfgpu_cross_term_dev(h, W1.data_ptr(), uX1.data_ptr(), W2.data_ptr(), uX2.data_ptr(), T.data_ptr())))
        t_mv = cuda_timed(torch, lambda: _lib.check(lib.vdfgpu_multiply_vec_dev(h, W1.data_ptr(), uX1.data_ptr(), ABC.data_ptr())))
        # Spartan's inner sum-check table (SURVEY 8f rank 2): transposed product over the column view
        t_br = cuda_timed(torch, lambda: _lib.check(lib.vdfgpu_r1cs_bind_rows_dev(h, E1.data_ptr(), rr3.data_ptr(), ABC.data_ptr(), Mt.data_ptr())))
        out = {"coefficients": "A = +1, B = full-size random, C = +1 / -1" if mix == "random_B" else "all +1 / -1 (step-circuit mix)"}
        for name, t, b in (("cross_term", t_ct, b_ct), ("multiply_vec", t_mv, b_mv), ("bind_rows", t_br, b_br)):
            out[name] = {"ms": t * 1e3, "algorithmic_bytes": b, "achieved_gbs": b / t / 1e9, "frac_of_hbm": b / t / 1e9 / peak}
        res[mix] = out
        _lib.check(lib.vdfgpu_r1cs_destroy(h))
    t_fd = cuda_timed(torch, lambda: _lib.check(lib.vdfgpu_fold_dev(1, W1.data_ptr(), W2.data_ptr(), vars_, E1.data_ptr(), T.data_ptr(), cons, rr.data_ptr())))
    res["fold"] = {"ms": t_fd * 1e3, "algorithmic_bytes": b_fd, "achieved_gbs": b_fd / t_fd / 1e9, "frac_of_hbm": b_fd / t_fd / 1e9 / peak}
    return res


def cpu_fold_step(shape, W, X, sec_shape, sec_W, sec_X, gens, sec_gens, _lib):
    """CPU baseline leg: the same step through oracle/cpu_ref.c on all host cores."""
    from oracle import cpu_ref as C, pasta as O
    cores = C.ncores()
    lib = _lib.load()
    parts = []
    for curve, sh, w, x, g in ((0, shape, W, X, gens), (1, sec_shape, sec_W, sec_X, sec_gens)):
        fid, cons, nvars, io, A, B, Cm = sh
        m = O.MODULUS[fid]
        ngen = max(cons, nvars)
        pts = bytearray(72 * ngen)
        _lib.check(lib.vdfgpu_gens_export(g._h, 0, ngen, _lib.as_ptr(pts)))
        coo = O.shape_to_coo_bytes(O.R1CSShape(m, cons, nvars, io, A, B, Cm))
        parts.append((curve, fid, m, cons, nvars, io, O.fes_to_bytes(w, m), O.fes_to_bytes(x, m), bytes(pts), coo))
    best = None
    for _ in range(2):
        t0 = time.perf_counter()
        for curve, fid, m, cons, nvars, io, wb, xb, pts, coo in parts:
            one = O.fe_to_bytes(1, m)
            abc1 = C.multiply_vec(fid, cons, nvars, io, coo, wb, one, xb)
            abc2 = C.multiply_vec(fid, cons, nvars, io, coo, wb, one, xb)
            T = C.cross_term(fid, cons, abc1, abc2, one)
            C.msm(curve, pts[:72 * nvars], wb, True, cores)
            C.msm(curve, pts[:72 * cons], T, True, cores)
            r = O.fe_to_bytes(0x1234567890ABCDEF, m)
            C.fold(fid, wb, wb, r)
            C.fold(fid, T, T, r)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return {"fold_steps_per_s": 1.0 / best, "ms": best * 1e3, "cores": cores, "kind": "port"}


def nova_step_measurements(_lib, ts=(10, 100, 1000, 1024, 4096, 16384)):
    """GPU side of one Nova fold step = NIFS on the secondary curve (Vesta; SYNTHETIC 10.3k-constraint block, the
    trivial step circuit) followed by NIFS on the primary curve (Pallas; step circuit of t inverse-MinRoot rounds + a
    SYNTHETIC 9.8k-constraint augmented block): per curve the fresh witness goes H2D, cross-term, ONE batched MSM for
    commit(W2) and commit(T), commitments D2H, fold with the challenge.  t = 10 / 100 / 1000 are the reference's
    own bench parameters (benches/nova.rs:63-65, BASELINE config 1), t = 1024 / 4096 / 16384 BASELINE config 3.
    Three variants per t: normalised commitments; un-normalised Jacobian commitments (what pasta-msm returns; the
    caller's to_affine() normalises); and the latter with the 4t+1 step variables taken from the device-resident
    witness bank (SURVEY 8f rank 1) instead of the host.  bellperson synthesis and the Poseidon RO (host) are not timed."""
    from vdf_b200 import encoding as E, msm as G, nova as N, synthetic as S   # inputs: package-side generator
    res = {}
    s_cons, s_vars, s_io, sA, sB, sC, sec_W, sec_X = S.step_instance(E.FP, 0, 10300, seed=7)
    sec_gs = N.R1CSShape(E.FP, s_cons, s_vars, s_io, sA, sB, sC)
    sWb, sXb = E.fes_to_bytes(sec_W, E.P), E.fes_to_bytes(sec_X, E.P)
    sec_shape = (E.FP, s_cons, s_vars, s_io, sA, sB, sC)
    r_fixed = 0x1234567890ABCDEF
    reps = 15

    def timed(step):
        for _ in range(3):
            step()
        t0 = time.perf_counter()
        for _ in range(reps):
            step()
        return (time.perf_counter() - t0) / reps

    for t in ts:
        cons, nvars, io, A, B, C, W, X = S.step_instance(E.FQ, t, 9800, seed=42)
        shape = (E.FQ, cons, nvars, io, A, B, C)
        gs = N.R1CSShape(E.FQ, cons, nvars, io, A, B, C)
        Wb, Xb = E.fes_to_bytes(W, E.Q), E.fes_to_bytes(X, E.Q)
        per = 4 * t + 1
        off = nvars - per
        entry = {"primary_cons": cons, "primary_vars": nvars, "secondary_cons": s_cons,
                 "h2d_bytes_per_step": 32 * (nvars + io + s_vars + s_io) + 64,
                 "h2d_bytes_per_step_bank": 32 * (nvars - per + io + s_vars + s_io) + 64, "d2h_bytes_per_step": 4 * 96}
        for variant, raw in (("normalised", False), ("raw_jacobian", True)):
            sec_gens = G.Generators.progression(1, K0, D, max(s_cons, s_vars), table=True, raw_jacobian=raw)
            gens = G.Generators.progression(0, K0, D, max(cons, nvars), table=True, raw_jacobian=raw)
            sec, pri = N.RunningProver(sec_gs, sec_gens), N.RunningProver(gs, gens)
            sec.set_running(sec_W, [0] * s_cons, N.RelaxedR1CSInstance(None, None, list(sec_X), 1))
            pri.set_running(W, [0] * cons, N.RelaxedR1CSInstance(None, None, list(X), 1))

            rp = N.RecursiveProver(pri, sec)    # the public two-curve step (vdf_b200/nova.py)

            def step():
                rp.prove_step_bytes(sWb, sXb, Wb, Xb, r_fixed, r_fixed)

            dt = timed(step)
            if not raw:
                entry.update({"fold_steps_per_s": 1.0 / dt, "ms": dt * 1e3})
            else:
                entry.update({"raw_jacobian_fold_steps_per_s": 1.0 / dt, "raw_jacobian_ms": dt * 1e3})
                # f1: the step part of the witness comes from the device-resident bank (one state per step; the bench
                # folds the same step repeatedly, the bank holds 4 of them as a proof with 4 steps would)
                bank = N.WitnessBank(E.FQ, [tuple(W[off - 3:off])] * 4, t)
                holed = bytes(Wb[:32 * off]) + bytes(32 * per)
                k = [0]

                def step_bank():
                    rp.prove_step_bytes(sWb, sXb, holed, Xb, r_fixed, r_fixed, bank=bank, step=k[0] & 3, step_offset=off)
                    k[0] += 1

                dtb = timed(step_bank)
                entry.update({"bank_fold_steps_per_s": 1.0 / dtb, "bank_ms": dtb * 1e3})
                bank.close()
                # CPU restatement of the same step's data-parallel work on the host cores (oracle/cpu_ref.c, "port");
                # after every GPU variant: 16 busy host threads disturb the next wall-clock measurement for a while
                try:
                    entry["cpu_port"] = cpu_fold_step(shape, W, X, sec_shape, sec_W, sec_X, gens, sec_gens, _lib)
                except Exception as e:
                    entry["cpu_port"] = {"error": repr(e)}
            pri.close(); sec.close(); gens.close(); sec_gens.close()
        gs.close()
        res[str(t)] = entry
    sec_gs.close()
    res["note"] = ("GPU side only; augmented-circuit blocks are SYNTHETIC; host synthesis and Poseidon RO not timed; wall clock "
                   "around the C-ABI calls (vdfgpu_running_commit[_step] + vdfgpu_running_finish per curve), host witness in, commitments out")
    return res


def minroot_verify_measurements(lib, _lib, torch, n=1 << 16, ts=(10, 1000, 10000)):
    """Batched verification (SURVEY 8d C4; t = 10 000 is benches/vdf.rs:26): 2^16 independent chains, originals
    computed by inverse_eval, a fixed 1 % corrupted; the verdict pattern is checked inside the bench."""
    import numpy as np
    out = {}
    gen = torch.Generator(device="cuda")
    gen.manual_seed(7)
    res = torch.randint(0, 1 << 62, (n, 12), dtype=torch.int64, device="cuda", generator=gen)
    res[:, 3::4] &= (1 << 61) - 1                      # every element < 2^253 < modulus
    res_h = res.cpu().numpy()
    bad = np.arange(n) % 100 == 37
    for t in ts:
        orig_h = np.zeros_like(res_h)
        _lib.check(lib.vdfgpu_minroot_inverse_eval_batch(1, res_h.ctypes.data, t, n, orig_h.ctypes.data))
        orig_h[bad, 0] ^= 1                              # corrupt x of 1 % of the originals
        orig = torch.from_numpy(orig_h).cuda()
        ok = torch.zeros(n, dtype=torch.uint8, device="cuda")
        fn = lib.vdfgpu_minroot_check_batch_dev
        reps = 5 if t <= 1000 else 2
        s = cuda_timed(torch, lambda: _lib.check(fn(1, res.data_ptr(), orig.data_ptr(), None, t, n, ok.data_ptr())), reps=reps, warm=1)
        verdict_ok = bool((ok.cpu().numpy() == (~bad).astype(np.uint8)).all())
        ok_h = np.zeros(n, dtype=np.uint8)
        t0 = time.perf_counter()
        _lib.check(lib.vdfgpu_minroot_check_batch(1, res_h.ctypes.data, orig_h.ctypes.data, None, t, n, ok_h.ctypes.data))
        e2e_s = time.perf_counter() - t0
        out[str(t)] = {"value": n * t / s, "unit": "MinRoot steps verified/s", "ms": s * 1e3, "chains": n, "t": t,
                       "corrupted_fraction": float(bad.mean()), "verdicts_correct": verdict_ok and bool((ok_h == (~bad)).all()),
                       "e2e_ms_host_states": e2e_s * 1e3, "e2e_value": n * t / e2e_s,
                       "mul32_per_step_convention": 3 * MUL32_PER_FIELD_MUL}
    return out


def dropin_measurements(lib, _lib, torch, sizes=(13904, 75344, 1 << 22)):
    """The literal pasta-msm symbol (what an unmodified nova-snark reaches): mult_pippenger_pallas with 72-byte host
    points and host scalars.  First call (uploads the points, builds the table), later calls (resident set), and
    vdfgpu_msm (explicit generator handle, synchronous) at the same size for comparison."""
    import numpy as np
    from vdf_b200 import msm as G
    out = {}
    rs = np.random.RandomState(3)
    for n in sizes:
        g = G.Generators.progression(0, K0, D, n, table=True)
        pts = np.zeros(72 * n, dtype=np.uint8)
        _lib.check(lib.vdfgpu_gens_export(g._h, 0, n, pts.ctypes.data))
        raw = rs.randint(0, 1 << 32, size=(n, 8), dtype=np.uint64).astype(np.uint32)
        raw[:, 7] &= 0x3FFFFFFF
        res, ref = np.zeros(96, dtype=np.uint8), np.zeros(96, dtype=np.uint8)
        _lib.check(lib.vdfgpu_dropin_cache_clear())

        def drop():
            lib.mult_pippenger_pallas(res.ctypes.data, pts.ctypes.data, n, raw.ctypes.data, True)

        def handle():
            _lib.check(lib.vdfgpu_msm(g._h, raw.ctypes.data, n, ref.ctypes.data))

        def wall(fn, reps):
            t0 = time.perf_counter()
            for _ in range(reps):
                fn()
            return (time.perf_counter() - t0) / reps * 1e3

        first = wall(drop, 1)
        second = wall(drop, 1)
        reps = 10 if n < (1 << 20) else 4
        steady = wall(drop, reps)
        handle(); handle()
        h_ms = wall(handle, reps)
        out[str(n)] = {"first_call_ms": first, "second_call_ms": second, "steady_ms": steady, "vdfgpu_msm_sync_ms": h_ms,
                       "steady_over_handle": steady / h_ms, "same_bytes_as_handle_path": bool((res == ref).all()),
                       "host_memory": "pageable (numpy), points 72 B + scalars 32 B per point"}
        g.close()
        _lib.check(lib.vdfgpu_dropin_cache_clear())
    out["note"] = "sample verification of the cached set (default VDFGPU_DROPIN_VERIFY=sample)"
    return out


def sumcheck_measurements(lib, _lib, torch, ell=24):
    """SURVEY 8f rank 2: the sum-check kernels of CompressedSNARK::prove on 2^24-entry tables (4 x 512 MiB, far beyond
    L2): the first (largest) round's evaluation and bind kernels against the HBM roofline, and a whole ell-round cubic
    sum-check with a trivial host callback (Nova's own tables have 2^14 - 2^17 entries and are launch-bound)."""
    n = 1 << ell
    tabs = [rand_fe_dev(torch, n) for _ in range(4)]
    peak, src = hbm_peak()
    r_host = (ctypes.c_uint64 * 4)(5, 0, 0, 0)
    calls = []

    def cb(_user, rnd, evals, n_evals, r_out):
        calls.append(rnd)
        ctypes.memmove(r_out, r_host, 32)
        return 0

    fn = _lib.ROUND_FN(cb)
    final = (ctypes.c_uint8 * 128)()
    # one round = evaluation (reads 4 tables) + bind (reads 4 tables, writes 4 half tables): time a 1-variable prefix
    # by running the full sum-check and dividing is not possible, so time whole sum-checks: bytes = sum over rounds
    reps = 3
    times = []
    for _ in range(reps + 1):
        fresh = [t.clone() for t in tabs]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _lib.check(lib.vdfgpu_sumcheck_cubic_dev(1, *[t.data_ptr() for t in fresh], ell, ctypes.cast(fn, ctypes.c_void_p), None, final))
        times.append(time.perf_counter() - t0)
        del fresh
    dt = min(times[1:])
    # algorithmic bytes: round k (length n / 2^k): evaluation reads 4 tables, bind reads 4 and writes 4 halves
    alg = sum(4 * 32 * (n >> k) + 4 * 32 * (n >> k) + 4 * 32 * (n >> (k + 1)) for k in range(ell))
    quad = [rand_fe_dev(torch, n) for _ in range(2)]
    t0 = time.perf_counter()
    _lib.check(lib.vdfgpu_sumcheck_quad_dev(1, quad[0].data_ptr(), quad[1].data_ptr(), ell, ctypes.cast(fn, ctypes.c_void_p), None, final))
    dq = time.perf_counter() - t0
    algq = sum(2 * 32 * (n >> k) * 2 + 2 * 32 * (n >> (k + 1)) for k in range(ell))
    # one IPA round's generator fold (CommitGens::fold): 2^16 outputs of r^-1 G_L + r G_R through the host API
    ipa = {}
    try:
        import numpy as np
        from vdf_b200 import msm as G
        m = 1 << 16
        g = G.Generators.progression(0, K0, D, 2 * m, table=False)
        pts = np.zeros(72 * 2 * m, dtype=np.uint8)
        _lib.check(lib.vdfgpu_gens_export(g._h, 0, 2 * m, pts.ctypes.data))
        g.close()
        w = np.frombuffer(os.urandom(64), dtype=np.uint8).copy()
        w[31] &= 0x3F; w[63] &= 0x3F
        outp = np.zeros(72 * m, dtype=np.uint8)
        for _ in range(2):
            t0 = time.perf_counter()
            _lib.check(lib.vdfgpu_points_lincomb(0, pts.ctypes.data, pts.ctypes.data + 72 * m, m, w.ctypes.data, w.ctypes.data + 32, outp.ctypes.data))
            di = time.perf_counter() - t0
        ipa = {"outputs": m, "ms": di * 1e3, "outputs_per_s": m / di,
               "note": "vdfgpu_points_lincomb, host points in and out (9.4 MB up, 4.7 MB down), two 255-bit scalars per output"}
    except Exception as e:
        ipa = {"error": repr(e)}
    rounds_cb = len(calls) // (reps + 2)
    # the same phases at the size of the largest Nova circuit (t = 16384: 59k constraints -> 2^16-entry outer tables,
    # 75k columns -> 2^17-entry inner tables): launch-bound there; tables are random (the time depends on sizes only),
    # the transposed product runs on the real step shape
    nova = {}
    try:
        from vdf_b200 import encoding as E, nova as N, synthetic as S
        cons, nvars, io, A, Bm, C, W, X = S.step_instance(E.FQ, 16384, 9800, seed=42)
        gs = N.R1CSShape(E.FQ, cons, nvars, io, A, Bm, C)
        ncols = nvars + 1 + io
        ex, ey = max(1, (cons - 1).bit_length()), max(1, (ncols - 1).bit_length())
        eqr, r3 = rand_fe_dev(torch, cons), rand_fe_dev(torch, 3)
        scratch = torch.zeros((3 * cons, 4), dtype=torch.int64, device="cuda")
        Mt = torch.zeros((1 << ey, 4), dtype=torch.int64, device="cuda")
        t_br = cuda_timed(torch, lambda: _lib.check(lib.vdfgpu_r1cs_bind_rows_dev(gs._h, eqr.data_ptr(), r3.data_ptr(), scratch.data_ptr(), Mt.data_ptr())))

        def wall(fn_, reps_=3):
            best = None
            for _ in range(reps_):
                torch.cuda.synchronize()
                t0_ = time.perf_counter()
                fn_()
                d_ = time.perf_counter() - t0_
                best = d_ if best is None or d_ < best else best
            return best

        def outer():
            tb = [rand_fe_dev(torch, 1 << ex) for _ in range(4)]
            torch.cuda.synchronize()
            t0_ = time.perf_counter()
            _lib.check(lib.vdfgpu_sumcheck_cubic_dev(1, *[t.data_ptr() for t in tb], ex, ctypes.cast(fn, ctypes.c_void_p), None, final))
            return time.perf_counter() - t0_

        def inner():
            tb = [rand_fe_dev(torch, 1 << ey) for _ in range(2)]
            torch.cuda.synchronize()
            t0_ = time.perf_counter()
            _lib.check(lib.vdfgpu_sumcheck_quad_dev(1, tb[0].data_ptr(), tb[1].data_ptr(), ey, ctypes.cast(fn, ctypes.c_void_p), None, final))
            return time.perf_counter() - t0_

        t_out = min(outer() for _ in range(4))
        t_in = min(inner() for _ in range(4))
        nova = {"t": 16384, "cons": cons, "cols": ncols, "outer_cubic_ms": t_out * 1e3, "outer_rounds": ex,
                "bind_rows_ms": t_br * 1e3, "inner_quad_ms": t_in * 1e3, "inner_rounds": ey,
                "note": "wall clock incl. one 96-byte read-back + trivial host callback per round; bind_rows by CUDA events"}
        gs.close()
    except Exception as e:
        nova = {"error": repr(e)}
    return {"ell": ell, "entries": n, "rounds_called_back": rounds_cb, "ipa_generator_fold": ipa, "nova_size": nova,
            "cubic": {"ms": dt * 1e3, "algorithmic_bytes": alg, "achieved_gbs": alg / dt / 1e9, "frac_of_hbm": alg / dt / 1e9 / peak,
                      "field_mul_per_s": 10 * n / dt},
            "quad": {"ms": dq * 1e3, "algorithmic_bytes": algq, "achieved_gbs": algq / dq / 1e9, "frac_of_hbm": algq / dq / 1e9 / peak},
            "hbm_peak_gbs": peak, "hbm_peak_source": src,
            "note": "wall clock of vdfgpu_sumcheck_*_dev on device-resident tables incl. one 96-byte D2H + host callback per round; "
                    "the cubic round does 6 multiplications per 256 bytes and is multiply-bound before it is HBM-bound"}


class MsmRunner:
    """n-point MSM on a device-resident generator set, device-resident scalars: serial and two-in-flight timings."""

    def __init__(self, torch, lib, _lib, n, k0=K0, raw=False, seed=42, table=True):
        from vdf_b200 import msm as G
        self.torch, self.lib, self._lib, self.n = torch, lib, _lib, n
        t0 = time.perf_counter()
        self.gens = G.Generators.progression(0, k0, D, n, table=table, raw_jacobian=raw)
        torch.cuda.synchronize()
        self.setup_s = time.perf_counter() - t0
        gen = torch.Generator(device="cuda")
        gen.manual_seed(seed)
        self.scal = rand_fe_dev(torch, n, gen)
        self.outs = [torch.zeros(96, dtype=torch.uint8, device="cuda") for _ in range(4)]
        self.streams = [torch.cuda.Stream() for _ in range(4)]

    def launch(self, slot):
        """enqueue one commitment on stream `slot` (each stream has its own workspace arena inside the library)"""
        s = self.streams[slot]
        self._lib.check(self.lib.vdfgpu_set_stream(s.cuda_stream))
        self._lib.check(self.lib.vdfgpu_msm_dev(self.gens._h, self.scal.data_ptr(), self.n, self.outs[slot].data_ptr()))
        return s

    def timed(self, steps, inflight, warm=2, after=None):
        """device time per step of `steps` commitments, `inflight` of them overlapping; `after(slot, stream)` is run
        behind every commitment on its stream (the multi-GPU combine)"""
        torch = self.torch
        ctx_stream = torch.cuda.current_stream()
        A, others = self.streams[0], self.streams[1:inflight]

        def run(count):
            for k in range(count):
                slot = k % inflight
                s = self.launch(slot)
                if after:
                    with torch.cuda.stream(s):
                        after(slot, s)

        run(max(warm, inflight) if warm else 0)     # every stream's workspace exists before the timed region
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(A)
        for s in others:
            s.wait_event(e0)
        run(steps)
        for s in others:
            ev = torch.cuda.Event()
            ev.record(s)
            A.wait_event(ev)
        e1.record(A)
        torch.cuda.synchronize()
        self._lib.check(self.lib.vdfgpu_set_stream(ctx_stream.cuda_stream))
        return e0.elapsed_time(e1) / steps

    def close(self):
        self.gens.close()


def sweep_measurements(lib, _lib, torch, log2s=(20, 22, 24, 26)):
    """Single-GPU size sweep (the metric names 2^20..2^26): device rate serial and two in flight, synchronous e2e from
    pinned host scalars, and the one-off cost of the generator set (progression + 2^(c w) table levels)."""
    out = {}
    for lg in log2s:
        n = 1 << lg
        try:
            r = MsmRunner(torch, lib, _lib, n)
            reps = 6 if lg <= 22 else (4 if lg == 24 else 3)
            ser = r.timed(reps, 1)
            deep = None
            if lg <= 24:       # several workspaces do not fit beside the 55 GB table of 2^26 points
                deep = r.timed(max(reps, 8), 4)
            _lib.check(lib.vdfgpu_trim())
            host = torch.empty((n, 4), dtype=torch.int64, pin_memory=True)
            host.copy_(r.scal)
            out_h = torch.zeros(96, dtype=torch.uint8, pin_memory=True)
            _lib.check(lib.vdfgpu_msm(r.gens._h, host.data_ptr(), n, out_h.data_ptr()))
            t0 = time.perf_counter()
            for _ in range(reps):
                _lib.check(lib.vdfgpu_msm(r.gens._h, host.data_ptr(), n, out_h.data_ptr()))
            e2e = (time.perf_counter() - t0) / reps
            out[str(lg)] = {"n": n, "window_bits": r.gens.window_bits(n), "affine_rounds": r.gens.affine_rounds(n),
                            "serial_ms": ser, "serial_gpoints_s": n / ser / 1e6,
                            "inflight4_ms": deep, "inflight4_gpoints_s": (n / deep / 1e6) if deep else None,
                            "sync_e2e_pinned_ms": e2e * 1e3, "sync_e2e_pinned_gpoints_s": n / e2e / 1e9,
                            "gens_setup_ms": r.setup_s * 1e3}
            r.close()
            del r, host
            _lib.check(lib.vdfgpu_trim())
            torch.cuda.empty_cache()
        except Exception as e:
            out[str(lg)] = {"error": repr(e)}
    return out


def gens_from_host_cost(lib, _lib, torch, log2n=22):
    """What a real PublicParams pays once per generator set (src/nova/proof.rs:232-237): 72-byte points uploaded from
    the host, repacked, 2^(c w) table levels built.  (Deriving the points themselves -- hash-to-curve -- is SURVEY 8f
    rank 3 and not built.)"""
    import numpy as np
    from vdf_b200 import msm as G
    n = 1 << log2n
    g = G.Generators.progression(0, K0, D, n, table=False)
    pts = np.zeros(72 * n, dtype=np.uint8)
    _lib.check(lib.vdfgpu_gens_export(g._h, 0, n, pts.ctypes.data))
    g.close()
    h = ctypes.c_void_p()
    t0 = time.perf_counter()
    _lib.check(lib.vdfgpu_gens_create(0, pts.ctypes.data, n, 1, 0, ctypes.byref(h)))
    dt = time.perf_counter() - t0
    _lib.check(lib.vdfgpu_gens_destroy(h))
    return {"log2n": log2n, "ms": dt * 1e3, "h2d_bytes": 72 * n, "host_memory": "pageable"}


def extra_measurements(lib, _lib, torch, args):
    out = {}
    for name, fn in (("nova_step", lambda: nova_step_measurements(_lib)),
                     ("minroot_verify", lambda: minroot_verify_measurements(lib, _lib, torch)),
                     ("r1cs_hbm", lambda: r1cs_hbm_measurements(lib, _lib, torch)),
                     ("dropin", lambda: dropin_measurements(lib, _lib, torch)),
                     ("sumcheck", lambda: sumcheck_measurements(lib, _lib, torch)),
                     ("gens_from_host", lambda: gens_from_host_cost(lib, _lib, torch))):
        try:
            t0 = time.perf_counter()
            out[name] = fn()
            out[name]["bench_wall_s"] = time.perf_counter() - t0
        except Exception as e:  # side measurement: never lose the headline line
            out[name] = {"error": repr(e)}
    if not args.no_sweep:
        try:
            t0 = time.perf_counter()
            out["sweep"] = sweep_measurements(lib, _lib, torch)
            out["sweep"]["bench_wall_s"] = time.perf_counter() - t0
        except Exception as e:
            out["sweep"] = {"error": repr(e)}
    return out


def strong_scaling(torch, dist, lib, _lib, rank, world, totals=(24, 26)):
    """Fixed total size split over the ranks by point range (SURVEY 8d C5): 2^24 and 2^26 points in all.  Rank 0 first
    times the whole problem alone (the same-run single-GPU figure), then every rank takes 1/world of it."""
    out = {}
    for lg in totals:
        total = 1 << lg
        n = total // world
        entry = {"points_total": total, "points_per_gpu": n}
        try:
            single = None
            if rank == 0:
                r1 = MsmRunner(torch, lib, _lib, total, raw=False)
                single = r1.timed(3, 1)
                r1.close()
                del r1
                _lib.check(lib.vdfgpu_trim())
                torch.cuda.empty_cache()
            dist.barrier()
            r = MsmRunner(torch, lib, _lib, n, k0=K0 + rank * n * D, raw=True, seed=1000 + rank)
            gathered = [torch.zeros(96 * world, dtype=torch.uint8, device="cuda") for _ in range(4)]
            total_dev = [torch.zeros(96, dtype=torch.uint8, device="cuda") for _ in range(4)]

            def combine(slot, s):
                dist.all_gather_into_tensor(gathered[slot], r.outs[slot])
                _lib.check(lib.vdfgpu_set_stream(s.cuda_stream))
                _lib.check(lib.vdfgpu_point_sum_dev(0, gathered[slot].data_ptr(), world, total_dev[slot].data_ptr()))

            res = {}
            deep = 4 if n <= (1 << 24) else 2
            for inflight in (1, deep):
                dist.barrier()
                ms = r.timed(6 if inflight == 1 else 8, inflight, after=combine)
                t = torch.tensor([ms], dtype=torch.float64, device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                res[inflight] = float(t.item())
            entry.update({"serial_ms": res[1], "serial_gpoints_s": total / res[1] / 1e6,
                          "inflight": deep, "inflight_ms": res[deep], "inflight_gpoints_s": total / res[deep] / 1e6})
            if rank == 0:
                entry["single_gpu_serial_ms"] = single
                entry["speedup_vs_single_gpu_serial"] = single / res[1]
                entry["efficiency_serial"] = single / res[1] / world
            r.close()
            del r
            _lib.check(lib.vdfgpu_trim())
            torch.cuda.empty_cache()
        except Exception as e:
            entry["error"] = repr(e)
        out[str(lg)] = entry
    return out


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from vdf_b200 import _lib
    from vdf_b200 import msm as G
    from vdf_b200.encoding import known_dlog_scalar

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world > 1:
        args.gpus = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the GPU path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = _lib.load()
    _lib.check(lib.vdfgpu_init(local_rank))
    # a dedicated (non-default) torch stream: torch.cuda.Event timing and the library's kernels share it.
    # (The legacy default stream has handle 0, which vdfgpu_set_stream reads as "use the library stream".)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    _lib.check(lib.vdfgpu_set_stream(stream.cuda_stream))

    n = 1 << args.log2n
    table = not args.plain
    steps, warmup = args.steps, max(3, args.warmup, args.inflight)   # every in-flight slot is warmed up at least once

    # generators: this rank's contiguous point range of the global progression; with several GPUs the partial results
    # stay un-normalised (one inversion after the combine instead of one per rank plus one)
    runner = MsmRunner(torch, lib, _lib, n, k0=K0 + rank * n * D, raw=world > 1, seed=42 + rank, table=table)
    gens, scal = runner.gens, runner.scal
    c_bits = gens.window_bits(n)
    W = (256 + c_bits - 1) // c_bits
    scal_host = torch.empty((n, 4), dtype=torch.int64, pin_memory=True)
    scal_host.copy_(scal)
    gathered = [torch.zeros(96 * world, dtype=torch.uint8, device="cuda") for _ in range(4)] if world > 1 else None
    total_dev = [torch.zeros(96, dtype=torch.uint8, device="cuda") for _ in range(4)]

    def combine(slot, s):
        dist.all_gather_into_tensor(gathered[slot], runner.outs[slot])
        _lib.check(lib.vdfgpu_set_stream(s.cuda_stream))
        _lib.check(lib.vdfgpu_point_sum_dev(0, gathered[slot].data_ptr(), world, total_dev[slot].data_ptr()))

    after = combine if world > 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- the timed region: K commitments, `inflight` of them overlapping ----
    runner.timed(warmup, args.inflight, warm=0, after=after)
    barrier()
    sampler = ClockSampler(visible_index(local_rank))
    if rank == 0:
        sampler.start()
    launches0 = lib.vdfgpu_launch_count()
    barrier()
    ms_per_step = max_over_ranks(runner.timed(steps, args.inflight, warm=0, after=after))
    barrier()
    launches = lib.vdfgpu_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    value = world * n / (ms_per_step * 1e-3) / 1e9
    if args.dump_outputs:   # the commitment the last timed step returned, before later passes reuse its buffer
        last = (steps - 1) % args.inflight
        last_out = (total_dev[last] if world > 1 else runner.outs[last]).cpu().numpy().tobytes()
    barrier()
    # the same K commitments one at a time on one stream (runs last: slot 0 then holds the final result)
    serial_ms = ms_per_step if args.inflight == 1 else max_over_ranks(runner.timed(steps, 1, warm=1, after=after))
    _lib.check(lib.vdfgpu_set_stream(stream.cuda_stream))

    # ---- parity of the (combined) commitment: known-discrete-log identity, every rank ----
    raw = scal.cpu().numpy().view(np.uint32).reshape(n, 8)
    mine = known_dlog_scalar(raw, K0, D, first=rank * n)
    if world > 1:
        blob = torch.frombuffer(bytearray(mine.to_bytes(80, "little")), dtype=torch.uint8).cuda()
        allb = torch.zeros(80 * world, dtype=torch.uint8, device="cuda")
        dist.all_gather_into_tensor(allb, blob)
        ab = allb.cpu().numpy().tobytes()
        mine = sum(int.from_bytes(ab[80 * r:80 * r + 80], "little") for r in range(world))
    expect_scalar = mine * pow(1 << 256, -1, Q_ORDER) % Q_ORDER        # scalars are Montgomery images
    g1 = G.Generators.progression(0, 1, 0, 1, table=False)            # the single point G
    expect = g1.commit_bytes((expect_scalar * (1 << 256) % Q_ORDER).to_bytes(32, "little"))
    g1.close()
    got = (total_dev[0] if world > 1 else runner.outs[0]).cpu().numpy().tobytes()   # slot 0 ran last (serial pass)
    parity_known_dlog = "ok" if got == expect else "MISMATCH"
    if parity_known_dlog != "ok":
        raise SystemExit(f"bench.py: rank {rank}: commitment differs from the known-discrete-log closed form")

    # ---- end to end through the C ABI with host buffers (wall clock, max over ranks) ----
    out_host = torch.zeros(96, dtype=torch.uint8, pin_memory=True)
    out_dev = torch.zeros(96, dtype=torch.uint8, device="cuda")

    def combine_host(src_host):
        out_dev.copy_(src_host, non_blocking=True)
        dist.all_gather_into_tensor(gathered[0], out_dev)
        _lib.check(lib.vdfgpu_point_sum_dev(0, gathered[0].data_ptr(), world, total_dev[0].data_ptr()))
        out_host.copy_(total_dev[0], non_blocking=True)

    def e2e_sync(host_ptr, k_steps):
        # the call a user of the reference makes: commit(scalars) with HOST buffers, one call at a time
        barrier()
        t0 = time.perf_counter()
        for _ in range(k_steps):
            _lib.check(lib.vdfgpu_msm(gens._h, host_ptr, n, out_host.data_ptr()))
            if world > 1:
                combine_host(out_host)
                torch.cuda.synchronize()
        barrier()
        return max_over_ranks((time.perf_counter() - t0) / k_steps)

    e2e_sync(scal_host.data_ptr(), 2)
    sync_pinned_s = e2e_sync(scal_host.data_ptr(), steps)
    pageable = scal_host.numpy().copy()                       # ordinary malloc'ed memory, what a Rust Vec is
    e2e_sync(pageable.ctypes.data, 1)
    sync_pageable_s = e2e_sync(pageable.ctypes.data, max(3, steps // 2))
    # the asynchronous form of the same call, `depth` commitments in flight: every step still uploads its own n*32
    # bytes from pinned host memory and reads its own 96-byte result back, but the upload and the latency-bound stages
    # of one step run under the kernels of the others.  Independent commitments (the microbenchmark's case) allow
    # this; the serial MSMs of one Nova step do not, which is why all three numbers are reported.
    depth = max(2, args.inflight)
    outs = [torch.zeros(96, dtype=torch.uint8, pin_memory=True) for _ in range(depth)]

    def finish(slot):
        _lib.check(lib.vdfgpu_msm_wait(slot))
        if world > 1:
            combine_host(outs[slot])

    def pipelined(k_steps):
        for k in range(k_steps):
            if k >= depth:
                finish(k % depth)
            _lib.check(lib.vdfgpu_msm_submit(gens._h, scal_host.data_ptr(), n, outs[k % depth].data_ptr(), k % depth))
        for k in range(max(0, k_steps - depth), k_steps):
            finish(k % depth)

    pipelined(2 * depth)
    barrier()
    t0 = time.perf_counter()
    pipelined(steps)
    barrier()
    e2e_s = max_over_ranks((time.perf_counter() - t0) / steps)
    if world == 1 and bytes(outs[0].numpy().tobytes()) != bytes(out_host.numpy().tobytes()):
        raise SystemExit("bench.py: pipelined and synchronous commitments differ")
    e2e = {"value": world * n / e2e_s / 1e9, "unit": "Gpoints/s", "ms_per_step": e2e_s * 1e3,
           "h2d_bytes_per_step": n * 32, "d2h_bytes_per_step": 96,
           "api": f"vdfgpu_msm_submit / vdfgpu_msm_wait (pinned host scalars in, host point out), {depth} commitments in flight",
           "sync_pinned": {"value": world * n / sync_pinned_s / 1e9, "ms_per_step": sync_pinned_s * 1e3,
                           "api": "vdfgpu_msm(gens, pinned host scalars, n, host out), one call at a time"},
           "sync_pageable": {"value": world * n / sync_pageable_s / 1e9, "ms_per_step": sync_pageable_s * 1e3,
                             "api": "vdfgpu_msm(gens, pageable host scalars (what a Rust Vec is), n, host out), one call at a time"}}

    # ---- per-stage device time of the dominant kernel (CUDA events inside the library, same stream, serial) ----
    stage_names = ["digits", "scan", "scatter", "accumulate", "records", "reduce", "final"]
    _lib.check(lib.vdfgpu_profile_enable(1))
    acc = [0.0] * 7
    prof_reps = 3
    for _ in range(prof_reps):
        _lib.check(lib.vdfgpu_msm_dev(gens._h, scal.data_ptr(), n, runner.outs[0].data_ptr()))
        buf = (ctypes.c_double * 7)()
        _lib.check(lib.vdfgpu_profile_read(buf, 7))
        acc = [a + b for a, b in zip(acc, buf)]
    _lib.check(lib.vdfgpu_profile_enable(0))
    stage_ms = {k: v / prof_reps for k, v in zip(stage_names, acc)}

    strong = None
    if world > 1 and not args.no_extra and not args.no_sweep:
        runner_keep = (gens, scal)   # noqa: F841  (the weak-scaling set stays resident: 3.4 GB)
        strong = strong_scaling(torch, dist, lib, _lib, rank, world)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # integer-multiply roofline of the dominant kernel (bucket accumulation)
    pw, pl, pa = ctypes.c_double(), ctypes.c_double(), ctypes.c_double()
    _lib.check(lib.vdfgpu_imad_peak(ctypes.byref(pw), ctypes.byref(pl), ctypes.byref(pa)))
    alg_mul32 = float(n) * W * FIELD_MUL_PER_MADD * MUL32_PER_FIELD_MUL
    acc_s = stage_ms["accumulate"] * 1e-3
    R = gens.affine_rounds(n)
    traffic = None
    tfile = ROOT / "profiles" / "traffic.json"   # dram bytes of one accumulate stage from the committed ncu capture
    if tfile.exists():
        t = json.loads(tfile.read_text())
        if t.get("log2n") == args.log2n and t.get("window_bits") == c_bits and t.get("layout") == ("table" if table else "plain") \
                and t.get("affine_rounds", 0) == R:
            traffic = t.get("accumulate_stage_dram_bytes", t.get("accumulate_dram_bytes_per_launch"))
    # field multiplications the accumulate stage really executes: R batched-affine halving rounds at 6 per addition
    # (the list shrinks to ~E / 2^R), then the XYZZ mixed additions of what is left at 10
    E = float(n) * W
    left = E / (1 << R)
    executed_mul = (E - left) * 6 + left * FIELD_MUL_PER_MADD
    roofline = {
        "bound": "imad",
        "kernel": (f"accumulate stage = {R} batched-affine halving rounds (AffineFwdFn, BatchInvFn, AffineBwdFn) + "
                   "AccumulateFn (XYZZ ranges)") if R else "AccumulateFn (XYZZ bucket accumulation)",
        "achieved": alg_mul32 / acc_s / 1e12, "peak": pw.value / 1e12, "unit": "Tmul32/s",
        "frac": (alg_mul32 / acc_s) / pw.value, "traffic": traffic,
        "frac_executed": (executed_mul * 88 / acc_s) / pw.value,
        "algorithmic": f"n * W(c) * 10 field-mul * 136 mul32 (SURVEY 8d) with the real c={c_bits}, W={W}",
        "peak_source": "measured in this run: vdfgpu_imad_peak, register-only IMAD.WIDE.U32.X carry chains with loop-variant "
                       "multiplicands (nominal 148 SM x 4 SMSP x 8 lanes x 1.965 GHz = 9.3 T; MEASURED_PEAKS.json has no integer figure)",
        "frac_executed_note": "products really executed: 88 per field multiplication (the SURVEY convention counts 136), 6 "
                              "multiplications per affine addition and 10 per XYZZ addition; frac > 1 means the stage does "
                              "less arithmetic than the convention assumes",
        "measured": "stage times by CUDA events inside the library, one MSM at a time (the timed region overlaps stages of different MSMs)",
        "affine_rounds": R,
        "hbm_view": hbm_view(n, acc_s, traffic),
        "imad_lo_per_s": pl.value, "iadd3_per_s": pa.value,
        "kernel_ms": stage_ms["accumulate"], "stage_ms": stage_ms,
        "share_of_step": stage_ms["accumulate"] / max(1e-9, sum(stage_ms.values())),
        "judge_convention_c16_achieved": float(n) * 21760 / acc_s / 1e12,
        "whole_step_executed_frac": (executed_mul * 88 / (ms_per_step * 1e-3)) / pw.value,
    }

    cpu_baseline = None
    parity = None
    if world == 1:
        # the CPU restatement on the SAME points and scalars (full n), and byte parity of the commitment against it
        # (the only place bench.py executes oracle/)
        pts_bytes = bytearray(72 * n)
        _lib.check(lib.vdfgpu_gens_export(gens._h, 0, n, _lib.as_ptr(pts_bytes)))
        sc_bytes = scal_host.numpy().tobytes()
        cpu_baseline, cpu_out = cpu_msm_timed(bytes(pts_bytes), sc_bytes)
        parity = "ok" if bytes(out_host.numpy().tobytes()) == cpu_out else "MISMATCH"
        del pts_bytes, sc_bytes

    cfg = workload_config(args.log2n, world)
    line = {
        "metric": METRIC, "value": value, "unit": "Gpoints/s", "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32 limbs (255-bit Montgomery, exact)", "data": "synthetic",
        "config": cfg,
        "plan": {"inflight": args.inflight, "layout": "table" if table else "plain", "window_bits": c_bits, "windows": W, "affine_rounds": R,
                 "scalars": "uniform 254-bit, seed 42+rank", "points": "known-dlog progression generated on the device",
                 "gens_setup_ms": runner.setup_s * 1e3},
        "serial": {"value": world * n / (serial_ms * 1e-3) / 1e9, "ms_per_step": serial_ms,
                   "note": "one commitment at a time on one stream (what the serial MSMs of one Nova step see)"},
        "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
        "cpu_baseline": cpu_baseline, "parity_vs_cpu_full_size": parity, "parity_known_dlog_all_ranks": parity_known_dlog,
    }
    if strong is not None:
        line["extra"] = {"strong": strong}
    if not args.no_extra and world == 1:
        runner.close()
        _lib.check(lib.vdfgpu_trim())
        torch.cuda.empty_cache()
        line["extra"] = extra_measurements(lib, _lib, torch, args)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"commitment": last_out})
    print_json(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    # Exactly ONE line on stdout: libraries (NCCL's version banner, torchrun notices) write to fd 1 too, so
    # route fd 1 to stderr for the duration of the run and emit the JSON line on the saved descriptor.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    captured = []

    def emit(line):
        captured.append(line)

    global print_json
    print_json = emit
    try:
        if args.impl == "reference":
            run_reference(args)
        else:
            run_ours(args)
    finally:
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        for line in captured:
            os.write(1, (line + "\n").encode())
        os.close(real_stdout)


if __name__ == "__main__":
    main()
