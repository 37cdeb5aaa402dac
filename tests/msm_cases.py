"""Scalar families that reach each branch of the MSM's signed-digit recoding (DigitsFn in msm.cuh), oracle side.

DigitsFn reads a scalar in W = ceil(256 / c) windows of c bits and adds the carry of the window below: a value
raw > B = 2^(c-1) becomes the digit raw - 2^c and carries one into the next window.  Its three branches are a digit
of +B (no carry), a negative digit with a carry, and raw = 2^c after a carry (digit 0, carry on).  Uniform scalars
reach the last branch with probability about 2^-c per window, so at large c the families below are the only inputs
that run it."""
import numpy as np

from oracle import pasta as O


def signed_digits(v: int, c: int):
    """DigitsFn's recoding of v: (digits, carry_in) over W = ceil(256 / c) windows."""
    W, B, full = (256 + c - 1) // c, 1 << (c - 1), 1 << c
    digits, carry_in, carry = [], [], 0
    for w in range(W):
        raw = ((v >> (w * c)) & (full - 1)) + carry
        carry_in.append(carry)
        if raw > B:
            digits.append(raw - full)
            carry = 1
        else:
            digits.append(raw)
            carry = 0
    assert carry == 0, "a carry left the top window"
    assert sum(d << (w * c) for w, d in enumerate(digits)) == v
    return digits, carry_in


def one_digit(c: int, d: int) -> int:
    """d in every window below bit 254: in the table layout every entry of the scalar lands in bucket d."""
    return sum(d << (c * w) for w in range(254 // c))


def alt_sign(c: int, d: int) -> int:
    """Digit -d in windows 0..K-2 and +d in window K-1 (K = 254 // c); 0 < d < 2^(c-1)."""
    K = 254 // c
    return (d << (c * (K - 1))) - sum(d << (c * w) for w in range(K - 1))


def families(c: int, order: int):
    """Named scalar values v < order for window size c (the values DigitsFn sees after from_mont)."""
    K, B = 254 // c, 1 << (c - 1)
    fam = {
        "top_bucket": sum(B << (c * w) for w in range(K)),
        "neg_chain": sum((B + 1) << (c * w) for w in range(K)),
        "zero_with_carry": (1 << (c * K)) - 1,
        "zero_with_carry_254": (1 << 254) - 1,
        "order-1": order - 1,
        "order-2": order - 2,
        "half": (order - 1) // 2,
        "2^253": 1 << 253,
        "2^254-B": (1 << 254) - B,
        "zero": 0,
        "one": 1,
    }
    for d in sorted({1, B - 1, B}):
        fam[f"one_digit_{d}"] = one_digit(c, d)
    for d in sorted({1, B - 1}):
        fam[f"alt_sign_{d}"] = alt_sign(c, d)
    assert all(0 <= v < order for v in fam.values())
    return fam


def tiled(c: int, order: int, n: int, seed: int):
    """n scalars: the families of c tiled, every other slot a uniform value (0 and 1 are families)."""
    vals = list(families(c, order).values())
    rng = np.random.RandomState(seed)
    out = []
    for i in range(n):
        if i % 2 == 0:
            out.append(vals[(i // 2) % len(vals)])
        else:
            out.append(int.from_bytes(rng.bytes(32), "little") % order)
    return out


def limbs(values):
    """(len, 8) uint32 little-endian limbs of non-negative integers < 2^256."""
    return np.frombuffer(b"".join(v.to_bytes(32, "little") for v in values), dtype=np.uint32).reshape(-1, 8)


def tile_index(n: int, k: int, seed: int):
    """n indices into a table of k distinct scalars, in a seeded order."""
    return np.random.RandomState(seed).randint(0, k, size=n)


def mont_table(values, order: int) -> np.ndarray:
    """(len, 32) uint8 Montgomery encodings: tile large scalar vectors by indexing this table."""
    return np.frombuffer(O.fes_to_bytes(values, order), dtype=np.uint8).reshape(-1, 32)
