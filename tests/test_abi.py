"""CPU: the C-ABI library loads and exports every symbol include/vdfgpu.h declares; the ctypes table covers
them all; without a GPU compute calls fail loudly (no CPU fallback)."""
import re
from pathlib import Path

import pytest

from vdf_b200 import _lib

HEADER = Path(__file__).resolve().parent.parent / "include" / "vdfgpu.h"


def _declared():
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    return sorted(set(re.findall(r"\b((?:vdfgpu_|mult_pippenger_)\w+)\s*\(", text)))


def test_header_symbols_exported_and_bound():
    names = _declared()
    assert len(names) >= 30
    lib = _lib.load()
    for n in names:
        assert hasattr(lib, n), f"{n} declared in vdfgpu.h but not exported"
        assert n in _lib.PROTOTYPES, f"{n} has no ctypes prototype"
    assert sorted(_lib.PROTOTYPES) == names


def test_version_and_no_cpu_fallback():
    import torch
    lib = _lib.load()
    assert b"sm_100a" in lib.vdfgpu_version()
    if torch.cuda.is_available():
        pytest.skip("GPU present: the failure path is only observable without one")
    assert lib.vdfgpu_device_count() == 0
    assert lib.vdfgpu_init(0) == -2
    assert b"no CPU fallback" in lib.vdfgpu_last_error()
    from vdf_b200 import minroot as M, VdfGpuError
    with pytest.raises(VdfGpuError):
        M.PallasVDF().check(M.State(1, 2, 3), 1, M.State(1, 2, 3))


def test_encoding_roundtrip():
    from vdf_b200 import encoding as E
    from oracle import pasta as O
    for m in (E.P, E.Q):
        for v in (0, 1, m - 1, 1 << 200):
            assert E.fe_to_bytes(v, m) == O.fe_to_bytes(v, m)
            assert E.fe_from_bytes(E.fe_to_bytes(v, m), m) == v
    assert E.P == O.P and E.Q == O.Q
    pt = O.PALLAS.mul(5, O.PALLAS.gen)
    assert E.affine_to_bytes(pt, E.P) == O.affine_to_bytes(O.PALLAS, pt)
    assert E.point_from_bytes(O.jac_to_bytes(O.PALLAS, pt), E.P) == pt


def test_point_normalise_host_matches_oracle():
    """The host-side normalisation the host entry points apply to their results (vdfgpu_point_normalise_host, no GPU
    needed): (X, Y, Z) -> (X / Z^2, Y / Z^3, 1) byte for byte, identity -> zeros, already-normalised unchanged."""
    from oracle import pasta as O
    lib = _lib.load()
    rng = O.XorShiftRng()
    for cv in (O.PALLAS, O.VESTA):
        m = cv.base
        # Z per point, None = random: 20 points led by a normalised one, then the identity; then 25 points with
        # Z = 1 and Z = 0 interleaved among un-normalised ones
        for zs in ([1] + [None] * 19 + [0], [(None, 1, None, 0, None)[k % 5] for k in range(25)]):
            buf, want = bytearray(), bytearray()
            for z in zs:
                if z == 0:      # the identity, whatever X and Y hold
                    buf += O.fe_to_bytes(5, m) + O.fe_to_bytes(7, m) + bytes(32)
                    want += bytes(96)
                    continue
                pt = cv.mul(O.field_random(rng, cv.order), cv.gen)
                z = O.field_random(rng, m) if z is None else z
                buf += O.fe_to_bytes(pt[0] * z * z, m) + O.fe_to_bytes(pt[1] * z * z * z, m) + O.fe_to_bytes(z, m)
                want += O.jac_to_bytes(cv, pt)
            assert lib.vdfgpu_point_normalise_host(cv.cid, _lib.as_ptr(buf), len(zs)) == 0
            assert bytes(buf) == bytes(want)
    assert lib.vdfgpu_point_normalise_host(7, None, 0) == -1
