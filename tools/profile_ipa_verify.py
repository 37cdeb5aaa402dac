#!/usr/bin/env python
"""Batch verification of inner-product arguments (vdfgpu_ipa_verify_batch) on the device.  Per (curve, ell) in
PALLAS 14, 17, 20 and VESTA 17, on a table-layout progression set of 2^ell + 1 points, for k = 1, 8, 64 proofs:
  call_ms            wall time of one vdfgpu_ipa_verify_batch call (arguments encoded beforehand), ending in the
                     library's own wait; median and min over the runs after warm-up
  gens_hat_k_ms      k calls of vdfgpu_ipa_gens_hat with the same challenges: the device work a verifier has without
                     the batch call (one MSM per proof, and no device path for the fold of P)
  kernels_us         device time per call of IpaHalfTablesFn and IpaBatchScalarsFn: the kernel records of
                     torch.profiler (CUPTI), not CUDA events, in a pass of its own (3 calls)
  failing_k8_ms      (k = 8) the call with one invalid proof: the batch, then the single-proof checks in chunks of 4
Once, at PALLAS ell = 20 and k = 64, the host's share of a call:
  host_prep_ms       in a passing call, from its start to its first device allocation, copy or launch (CPU
                     timestamps of the torch.profiler trace around 3 calls): every host step before the device work --
                     the argument checks, the coordinate and curve checks, the batched inversions of Z and of r, the
                     scalars of both MSMs
  host_checks_ms     a call in which every proof is rejected by its last point (off the curve) after all its points
                     were checked, with comm_a un-normalised (Z != 1): the coordinate checks, the batched Z inversion
                     and the curve checks alone, with no device work
The proofs are synthetic and valid: random L_j = l_j G, R_j = rho_j G, challenges and scalars, and comm_a chosen to
satisfy the equation, a_hat G_hat + u_scale (a_hat b_hat - c) U0 - sum_j (r_j^2 L_j + r_j^-2 R_j), with G_hat from
vdfgpu_ipa_gens_hat.  The work of a call does not depend on how the proofs were made.
Writes one JSON line (default profiles/r3_ipa_verify.json) with the device name, power limit and max SM clock read in
the same run."""
import argparse
import json
import random
import statistics
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

K0, D = 1234567, 89


def stats(ts):
    return {"median": statistics.median(ts), "min": min(ts), "runs": len(ts)}


def synthetic_proofs(g, cv, ell, k, seed):
    from oracle import pasta as O
    from vdf_b200 import spartan as SP
    m = cv.order
    py = random.Random(seed)
    u0_log = (K0 + (1 << ell) * D) % m
    out = []
    for _ in range(k):
        rs = [py.randrange(1, m) for _ in range(ell)]
        ls = [py.randrange(1, m) for _ in range(ell)]
        ps = [py.randrange(1, m) for _ in range(ell)]
        a_hat, b_hat, c, u_scale = (py.randrange(1, m) for _ in range(4))
        G_hat = O.jac_from_bytes(cv, SP.ipa_gens_hat(g, rs))
        log = u_scale * (a_hat * b_hat - c) * u0_log
        for r, l_, p_ in zip(rs, ls, ps):
            log -= r * r * l_ + pow(r, -2, m) * p_
        comm = cv.add(cv.mul(a_hat, G_hat), cv.mul(log % m, cv.gen))
        pt = lambda x: O.jac_to_bytes(cv, cv.mul(x, cv.gen))  # noqa: E731
        out.append(([pt(x) for x in ls], [pt(x) for x in ps], rs, a_hat, O.jac_to_bytes(cv, comm), c, b_hat, u_scale))
    return out


class Call:
    """one vdfgpu_ipa_verify_batch call with its arguments encoded once"""

    def __init__(self, lib, _lib, g, cv, ell, proofs, comm=None, Ls=None):
        from oracle import pasta as O
        m = cv.order
        col = lambda i: O.fes_to_bytes([p[i] for p in proofs], m)  # noqa: E731
        self.keep = [comm or b"".join(p[4] for p in proofs), Ls or (b"".join(x for p in proofs for x in p[0]) or bytes(96)),
                     b"".join(x for p in proofs for x in p[1]) or bytes(96),
                     O.fes_to_bytes([r for p in proofs for r in p[2]], m) or bytes(32), col(3), col(5), col(6), col(7),
                     O.fes_to_bytes([random.randrange(1, m) for _ in proofs], m)]
        self.ok = bytearray(len(proofs))
        self.args = [g._h, ell, len(proofs)] + [_lib.as_ptr(b) for b in self.keep] + [_lib.as_ptr(self.ok)]
        self.fn, self.check = lib.vdfgpu_ipa_verify_batch, _lib.check

    def __call__(self):
        self.check(self.fn(*self.args))
        return list(self.ok)


def timed(fn, runs, warm):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(runs):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return stats(ts)


def kernel_us(torch, fn, calls=3):
    """device time per call of the two scalar-table kernels (torch.profiler, CUDA activities)"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {"timer": "torch.profiler kernel records (CUPTI)", "IpaHalfTablesFn": 0.0, "IpaBatchScalarsFn": 0.0}
    for e in prof.key_averages():
        for name in ("IpaHalfTablesFn", "IpaBatchScalarsFn"):
            if name in e.key:
                out[name] += e.device_time_total / calls
    return out


def measure(lib, _lib, torch, cid, ell, runs, warm, host_probe):
    from oracle import pasta as O
    from vdf_b200 import msm as G
    from vdf_b200 import spartan as SP
    cv = O.CURVES[cid]
    n = 1 << ell
    g = G.Generators.progression(cid, K0, D, n + 1, table=True)
    proofs = synthetic_proofs(g, cv, ell, 64, 1000 + ell + cid)
    res = {"curve": "pallas" if cid == 0 else "vesta", "ell": ell, "n": n, "by_k": []}
    for k in (1, 8, 64):
        call = Call(lib, _lib, g, cv, ell, proofs[:k])
        assert call() == [1] * k, "the synthetic proofs must verify"
        r = {"k": k, "call_ms": timed(call, runs, warm)}
        r["gens_hat_k_ms"] = timed(lambda: [SP.ipa_gens_hat(g, p[2]) for p in proofs[:k]], max(3, runs // 2), 1)
        r["kernels_us"] = kernel_us(torch, call)
        if k == 8:
            bad = list(proofs[:8])
            p = bad[5]
            bad[5] = p[:3] + ((p[3] + 1) % cv.order,) + p[4:]
            fail = Call(lib, _lib, g, cv, ell, bad)
            assert fail() == [int(q != 5) for q in range(8)]
            r["failing_k8_ms"] = timed(fail, runs, warm)
        print(json.dumps({"curve": res["curve"], "ell": ell, **r}), flush=True)
        res["by_k"].append(r)
    if host_probe:
        res["host_prep_ms"] = host_prep(torch, Call(lib, _lib, g, cv, ell, proofs))
        res["host_checks_ms"] = host_checks(lib, _lib, g, cv, ell, proofs, runs, warm)
    g.close()
    return res


DEVICE_WORK = ("cudaMallocAsync", "cudaMemcpyAsync", "cudaLaunchKernel", "cudaLaunchKernelExC", "cudaGraphLaunch")


def host_prep(torch, call, calls=3):
    """per call: the start of its record_function range to the first runtime call that enqueues device work"""
    from torch.profiler import ProfilerActivity, profile, record_function
    call()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            with record_function("ipa_verify_batch_call"):
                call()
    evs = prof.events()
    cpu = torch.autograd.DeviceType.CPU   # the range also appears as a GPU-side annotation: keep the host one
    ranges = sorted((e.time_range.start, e.time_range.end) for e in evs
                    if e.name == "ipa_verify_batch_call" and e.device_type == cpu)
    firsts, names = [], set()
    for t0, t1 in ranges:
        inside = sorted((e.time_range.start, e.name) for e in evs if e.name in DEVICE_WORK and t0 <= e.time_range.start <= t1)
        if inside:
            firsts.append((inside[0][0] - t0) / 1e3)
            names.add(inside[0][1])
    if not firsts:
        return {"method": "no runtime call recorded inside the call: not measured"}
    return {"method": "torch.profiler CPU timestamps, call start -> first " + "/".join(sorted(names)), **stats(firsts)}


def host_checks(lib, _lib, g, cv, ell, proofs, runs, warm):
    """every proof's last point (R_{ell-1}) off the curve, comm_a un-normalised: all points checked, nothing on the
    device"""
    from oracle import pasta as O
    p_ = cv.base
    comm = b""
    for p in proofs:
        x, y = O.jac_from_bytes(cv, p[4])
        z = 3
        comm += O.fe_to_bytes(x * z * z, p_) + O.fe_to_bytes(y * z ** 3, p_) + O.fe_to_bytes(z, p_)
    bad = []
    for p in proofs:
        Rs = list(p[1])
        x, y = O.jac_from_bytes(cv, Rs[-1])
        Rs[-1] = O.fe_to_bytes(x, p_) + O.fe_to_bytes(y + 1, p_) + O.fe_to_bytes(1, p_)
        bad.append((p[0], Rs) + p[2:])
    call = Call(lib, _lib, g, cv, ell, bad, comm=comm)
    launches = lib.vdfgpu_launch_count()
    assert call() == [0] * len(proofs)
    assert lib.vdfgpu_launch_count() == launches
    return {"k": len(proofs), **timed(call, runs, warm)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_ipa_verify.json"))
    ap.add_argument("--runs", type=int, default=7)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--configs", default="0:14,0:17,0:20,1:17", help="curve:ell list")
    args = ap.parse_args()
    import torch
    from profile_verify import device_info
    from vdf_b200 import _lib
    if not torch.cuda.is_available():
        raise SystemExit("profile_ipa_verify: no CUDA device (the measurement has no CPU fallback)")
    lib = _lib.load()
    _lib.check(lib.vdfgpu_init(0))
    res = {"device": device_info(), "configs": []}
    for spec in args.configs.split(","):
        cid, ell = (int(x) for x in spec.split(":"))
        res["configs"].append(measure(lib, _lib, torch, cid, ell, args.runs, args.warm, host_probe=(cid, ell) == (0, 20)))
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
