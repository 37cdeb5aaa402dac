#!/usr/bin/env python
"""The inner-product argument of CompressedSNARK::prove (spartan_with_ipa_pc [R]) on the device, at Nova sizes and
above.  Per (curve, ell) in PALLAS 10, 14, 17, 20 and VESTA 14, on a table-layout progression set of 2^ell + 1 points:
  prove_ms             wall time of vdfgpu_ipa_prove_dev (device vectors, consumed: re-copied before each run, outside
                       the timed window), ending in the library's own wait; median and min over the runs after warm-up
  prove_minus_cb_ms    the same minus the time spent inside the Python round callback (sha256 of L and R), timed in it
  round_msm_ms         per round j: the batched MSM (k = 2, n + 1 scalars with round j's zero pattern, raw results as the
                       round loop asks for them) timed alone with CUDA events, median over the runs
  gens_hat_ms          vdfgpu_ipa_gens_hat (host challenges in, normalised point out)
  block_path_ms        (ell = 10, 14) the per-round building blocks as tests/test_gpu_sumcheck.py's end-to-end IPA uses
                       them: host vectors, vdfgpu_inner_product x 2, mult_pippenger_* over the generator halves plus U
                       (a new host pointer every round), vdfgpu_vec_lincomb x 2, vdfgpu_points_lincomb
Writes one JSON line (default profiles/r3_ipa.json) with the device name, power limit and max SM clock read in the same
run."""
import argparse
import ctypes
import hashlib
import json
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


def random_fes(torch, n, seed):
    """n canonical field elements (values < 2^254 < both moduli) as a CUDA uint8 tensor of 32 n bytes"""
    g = torch.Generator().manual_seed(seed)
    t = torch.randint(0, 256, (n, 32), dtype=torch.uint8, generator=g)
    t[:, 31] &= 0x3F
    return t.reshape(-1).cuda()


def measure(lib, _lib, torch, cid, ell, runs, warm, block):
    """Everything on one caller stream: the library's work (vdfgpu_set_stream), the tensor copies and the CUDA events."""
    s = torch.cuda.Stream()
    _lib.check(lib.vdfgpu_set_stream(s.cuda_stream))
    try:
        with torch.cuda.stream(s):
            return measure_on_stream(lib, _lib, torch, cid, ell, runs, warm, block)
    finally:
        torch.cuda.synchronize()
        _lib.check(lib.vdfgpu_set_stream(None))


def measure_on_stream(lib, _lib, torch, cid, ell, runs, warm, block):
    from vdf_b200 import encoding as E, msm as G, spartan as SP
    order = E.CURVE_ORDER[cid]
    n = 1 << ell
    g = G.Generators.progression(cid, K0, D, n + 1, table=True)
    a0, b0 = random_fes(torch, n, 2 * ell + cid), random_fes(torch, n, 2 * ell + cid + 1)
    a, b = torch.empty_like(a0), torch.empty_like(b0)
    cb_s = [0.0]

    def challenge(rnd, L, R):
        t0 = time.perf_counter()
        r = int.from_bytes(hashlib.sha256(bytes([rnd]) + L + R).digest(), "little") % order or 1
        cb_s[0] += time.perf_counter() - t0
        return r

    walls, nets = [], []
    rs = None
    for k in range(warm + runs):
        a.copy_(a0)
        b.copy_(b0)
        torch.cuda.synchronize()
        cb_s[0] = 0.0
        t0 = time.perf_counter()
        _, _, rs, _ = SP.ipa_prove_dev(g, a, b, 3, challenge)
        wall = (time.perf_counter() - t0) * 1e3
        if k >= warm:
            walls.append(wall)
            nets.append(wall - cb_s[0] * 1e3)
    out = {"curve": "pallas" if cid == 0 else "vesta", "ell": ell, "n": n, "window_bits": g.window_bits(n + 1),
           "prove_ms": stats(walls), "prove_minus_cb_ms": stats(nets)}
    # per-round batched MSM, alone, on a raw-result set (the round loop's MSMs return raw Jacobian points)
    graw = G.Generators.progression(cid, K0, D, n + 1, table=True, raw_jacobian=True)
    S = random_fes(torch, n + 1, 7).view(n + 1, 32)
    idx = torch.arange(n + 1, device="cuda")
    outp = torch.empty(2 * 96, dtype=torch.uint8, device="cuda")
    lens = (ctypes.c_size_t * 2)(n + 1, n + 1)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    per_round = []
    for j in range(ell):
        m, h = n >> j, (n >> j) // 2
        left = ((idx % m) < h) & (idx < n)
        SL = torch.where(((idx % m) >= h).unsqueeze(1) | (idx == n).unsqueeze(1), S, 0).contiguous()
        SR = torch.where(left.unsqueeze(1) | (idx == n).unsqueeze(1), S, 0).contiguous()
        ptrs = (ctypes.c_void_p * 2)(SL.data_ptr(), SR.data_ptr())
        ts = []
        for k in range(warm + runs):
            ev0.record()
            _lib.check(lib.vdfgpu_msm_batch_dev(graw._h, ptrs, lens, 2, outp.data_ptr()))
            ev1.record()
            ev1.synchronize()
            if k >= warm:
                ts.append(ev0.elapsed_time(ev1))
        per_round.append(statistics.median(ts))
    out["round_msm_ms"] = per_round
    out["round_msm_sum_ms"] = sum(per_round)
    graw.close()
    ts = []
    for k in range(warm + runs):
        t0 = time.perf_counter()
        SP.ipa_gens_hat(g, rs)
        if k >= warm:
            ts.append((time.perf_counter() - t0) * 1e3)
    out["gens_hat_ms"] = stats(ts)
    if block:
        out["block_path_ms"] = block_path(lib, _lib, g, cid, ell, a0, b0, max(2, runs // 2))
    g.close()
    return out


def block_path(lib, _lib, g, cid, ell, a0, b0, runs):
    """All rounds on the host-vector building blocks; bytes stay bytes between the calls (no Python integers)."""
    from vdf_b200 import encoding as E
    order = E.CURVE_ORDER[cid]
    fid = E.CURVE_SCALAR_FIELD[cid]
    n = 1 << ell
    pts = bytearray(72 * (n + 1))
    _lib.check(lib.vdfgpu_gens_export(g._h, 0, n + 1, _lib.as_ptr(pts)))
    G0, U = bytes(pts[:72 * n]), bytes(pts[72 * n:])
    a_init, b_init = bytes(a0.cpu().numpy().tobytes()), bytes(b0.cpu().numpy().tobytes())
    pip = lib.mult_pippenger_pallas if cid == 0 else lib.mult_pippenger_vesta
    ts = []
    for k in range(1 + runs):
        a, b, Gb = a_init, b_init, G0
        t0 = time.perf_counter()
        m = n
        while m > 1:
            h = m // 2
            cL, cR = bytearray(32), bytearray(32)
            _lib.check(lib.vdfgpu_inner_product(fid, _lib.as_ptr(a[:32 * h]), _lib.as_ptr(b[32 * h:]), h, _lib.as_ptr(cL)))
            _lib.check(lib.vdfgpu_inner_product(fid, _lib.as_ptr(a[32 * h:]), _lib.as_ptr(b[:32 * h]), h, _lib.as_ptr(cR)))
            L, R = bytearray(96), bytearray(96)
            pip(_lib.as_ptr(L), _lib.as_ptr(Gb[72 * h:] + U), h + 1, _lib.as_ptr(a[:32 * h] + bytes(cL)), True)
            pip(_lib.as_ptr(R), _lib.as_ptr(Gb[:72 * h] + U), h + 1, _lib.as_ptr(a[32 * h:] + bytes(cR)), True)
            r = int.from_bytes(hashlib.sha256(bytes(L) + bytes(R)).digest(), "little") % order or 1
            rb, rib = E.fe_to_bytes(r, order), E.fe_to_bytes(pow(r, -1, order), order)
            a2, b2, G2 = bytearray(32 * h), bytearray(32 * h), bytearray(72 * h)
            _lib.check(lib.vdfgpu_vec_lincomb(fid, _lib.as_ptr(a[:32 * h]), _lib.as_ptr(a[32 * h:]), h, _lib.as_ptr(rb),
                                              _lib.as_ptr(rib), _lib.as_ptr(a2)))
            _lib.check(lib.vdfgpu_vec_lincomb(fid, _lib.as_ptr(b[:32 * h]), _lib.as_ptr(b[32 * h:]), h, _lib.as_ptr(rib),
                                              _lib.as_ptr(rb), _lib.as_ptr(b2)))
            _lib.check(lib.vdfgpu_points_lincomb(cid, _lib.as_ptr(Gb[:72 * h]), _lib.as_ptr(Gb[72 * h:]), h,
                                                 _lib.as_ptr(rib), _lib.as_ptr(rb), _lib.as_ptr(G2)))
            a, b, Gb = bytes(a2), bytes(b2), bytes(G2)
            m = h
        if k:
            ts.append((time.perf_counter() - t0) * 1e3)
    return stats(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_ipa.json"))
    ap.add_argument("--runs", type=int, default=7)
    ap.add_argument("--warm", type=int, default=2)
    ap.add_argument("--configs", default="0:10,0:14,0:17,0:20,1:14", help="curve:ell list")
    args = ap.parse_args()
    import torch
    from profile_verify import device_info
    from vdf_b200 import _lib
    if not torch.cuda.is_available():
        raise SystemExit("profile_ipa: no CUDA device (the measurement has no CPU fallback)")
    lib = _lib.load()
    _lib.check(lib.vdfgpu_init(0))
    res = {"device": device_info(), "configs": []}
    for spec in args.configs.split(","):
        cid, ell = (int(x) for x in spec.split(":"))
        r = measure(lib, _lib, torch, cid, ell, args.runs, args.warm, block=ell in (10, 14))
        print(json.dumps(r), flush=True)
        res["configs"].append(r)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
