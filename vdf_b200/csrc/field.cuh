// Pallas/Vesta base+scalar field arithmetic for sm_100a: 255-bit, 8 x 32-bit limbs, Montgomery
// form with R = 2^256 -- byte-identical to pasta_curves' Fp/Fq ([u64;4] little-endian limbs,
// SURVEY.md section 8a row a2; the reference uses them at src/minroot.rs:73-75,220-222,329-344).
//
// Both moduli are 2^254 + c with 32-bit limbs [1, M1, M2, M3, 0, 0, 0, 0x40000000] and
// -m^-1 mod 2^32 = 0xffffffff, so the Montgomery quotient digit is q = -t0 (no multiply) and a
// reduction row needs 3 real 32x32 products (M1, M2, M3) plus a shift for the 2^30 limb.
//
// Device path: PTX mad.lo.cc/madc.hi.cc chains laid out in even/odd columns so ptxas fuses every
// (lo, hi) pair into one IMAD.WIDE.U32(.X) with the carry in a predicate.  Host path (the library's host-side
// checks, normalisations and inversions, and the CPU emulation under tests/emul): plain C, the multiplier over
// 4 x 64-bit limbs with 128-bit products.
#pragma once
#include <cstdint>
#include <cstring>

#if defined(__CUDACC__)
#define VDF_HD __host__ __device__ __forceinline__
#define VDF_D __device__ __forceinline__
#else
#define VDF_HD inline
#define VDF_D inline
#endif

namespace vdf {

struct FpTag {  // Pallas base field / Vesta scalar field
  static constexpr uint32_t M1 = 0x992d30edu, M2 = 0x094cf91bu, M3 = 0x224698fcu;
  static constexpr int ID = 0;
};
struct FqTag {  // Pallas scalar field / Vesta base field
  static constexpr uint32_t M1 = 0x8c46eb21u, M2 = 0x0994a8ddu, M3 = 0x224698fcu;
  static constexpr int ID = 1;
};

#if defined(__CUDACC__)
// The modulus limbs M1..M3 as the multiplier reads them on the device.  They live in constant memory
// (uploaded by vdf::upload_field_constants() in every translation unit) instead of being immediates: with
// an immediate multiplicand ptxas splits each 32x32->64 multiply-add into IMAD (lo) + IMAD.HI (6
// multiply-pipe cycles per warp), with a uniform-register operand it emits one IMAD.WIDE.U32 (4 cycles).
static __constant__ uint32_t VDF_KMOD[2][4];

static inline cudaError_t upload_field_constants() {
  const uint32_t h[2][4] = {{FpTag::M1, FpTag::M2, FpTag::M3, 0x40000000u}, {FqTag::M1, FqTag::M2, FqTag::M3, 0x40000000u}};
  return cudaMemcpyToSymbol(VDF_KMOD, h, sizeof(h));
}
#endif

struct alignas(16) fe {
  uint32_t v[8];
};

template <class T>
struct Field {
  static constexpr uint32_t M1 = T::M1, M2 = T::M2, M3 = T::M3, M7 = 0x40000000u;

  static VDF_HD uint32_t mod_limb(int j) {
    return j == 0 ? 1u : j == 1 ? M1 : j == 2 ? M2 : j == 3 ? M3 : j == 7 ? M7 : 0u;
  }

  static VDF_HD fe zero() {
    fe r;
#pragma unroll
    for (int j = 0; j < 8; j++) r.v[j] = 0;
    return r;
  }

  // R mod m = 2^256 - 3m  (m is just above 2^254, so 3m < 2^256 < 4m): Montgomery form of 1.
  static VDF_HD fe one() {
    // computed at compile time by the host compiler / ptxas from the limbs
    fe r;
    uint64_t borrow = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) {
      uint64_t s = 3ull * mod_limb(j) + borrow;       // limb of 3m plus carry
      uint32_t lo = (uint32_t)s;
      borrow = s >> 32;
      r.v[j] = lo;
    }
    // r = 3m (fits 256 bits); now r = 2^256 - r = ~r + 1
    uint64_t c = 1;
#pragma unroll
    for (int j = 0; j < 8; j++) {
      uint64_t s = (uint64_t)(~r.v[j]) + c;
      r.v[j] = (uint32_t)s;
      c = s >> 32;
    }
    return r;
  }

  static VDF_HD bool is_zero(const fe& a) {
    uint32_t o = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) o |= a.v[j];
    return o == 0;
  }

  static VDF_HD bool eq(const fe& a, const fe& b) {
    uint32_t o = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) o |= a.v[j] ^ b.v[j];
    return o == 0;
  }

  // ---- add / sub / neg: inputs and outputs fully reduced in [0, m) -----------------------------
  static VDF_HD fe add(const fe& a, const fe& b) {
    fe s, t;
#if defined(__CUDA_ARCH__)
    add8(s.v, a.v, b.v);  // a+b < 2^256: no carry out
    uint32_t borrow = sub8_mod(t.v, s.v);
#else
    uint64_t c = 0;
    for (int j = 0; j < 8; j++) {
      c += (uint64_t)a.v[j] + b.v[j];
      s.v[j] = (uint32_t)c;
      c >>= 32;
    }
    int64_t bw = 0;
    for (int j = 0; j < 8; j++) {
      bw += (int64_t)s.v[j] - mod_limb(j);
      t.v[j] = (uint32_t)bw;
      bw >>= 32;
    }
    uint32_t borrow = (uint32_t)bw;
#endif
    fe r;
#pragma unroll
    for (int j = 0; j < 8; j++) r.v[j] = borrow ? s.v[j] : t.v[j];
    return r;
  }

  static VDF_HD fe sub(const fe& a, const fe& b) {
    fe d, t;
    uint32_t borrow;
#if defined(__CUDA_ARCH__)
    borrow = sub8(d.v, a.v, b.v);
    add8_mod(t.v, d.v);
#else
    int64_t bw = 0;
    for (int j = 0; j < 8; j++) {
      bw += (int64_t)a.v[j] - b.v[j];
      d.v[j] = (uint32_t)bw;
      bw >>= 32;
    }
    borrow = (uint32_t)bw;
    uint64_t c = 0;
    for (int j = 0; j < 8; j++) {
      c += (uint64_t)d.v[j] + mod_limb(j);
      t.v[j] = (uint32_t)c;
      c >>= 32;
    }
#endif
    fe r;
#pragma unroll
    for (int j = 0; j < 8; j++) r.v[j] = borrow ? t.v[j] : d.v[j];
    return r;
  }

  // a < m: the canonical range every arithmetic routine here assumes (pasta_curves' from_repr rejects the rest)
  static VDF_HD bool is_canonical(const fe& a) {
#if defined(__CUDA_ARCH__)
    fe t;
    return sub8_mod(t.v, a.v) != 0;   // a - m borrows
#else
    int64_t bw = 0;
    for (int j = 0; j < 8; j++) {
      bw += (int64_t)a.v[j] - mod_limb(j);
      bw >>= 32;
    }
    return bw != 0;
#endif
  }

  static VDF_HD fe neg(const fe& a) { return sub(zero(), a); }
  static VDF_HD fe dbl(const fe& a) { return add(a, a); }

  // ---- Montgomery multiplication ---------------------------------------------------------------
#if defined(__CUDA_ARCH__)
  // Every carry chain lives inside ONE asm statement: the compiler does not model the CC flag, so
  // a chain split over several statements could be reordered.
  // acc[j], acc[j+1] = a[j] * bi for j = 0, 2, 4, 6 (a is pre-offset by the caller)
  static VDF_D void mul_n(uint32_t* acc, const uint32_t* a, uint32_t bi) {
#pragma unroll
    for (int j = 0; j < 8; j += 2)
      asm("mul.lo.u32 %0, %2, %3; mul.hi.u32 %1, %2, %3;" : "=r"(acc[j]), "=r"(acc[j + 1]) : "r"(a[j]), "r"(bi));
  }
  // even[0] += odd[1];  odd = (odd >> 64) + a[0,2,4,6] * bi  (one chain; top pair is fresh)
  static VDF_D void shift_mad(uint32_t* even, uint32_t* odd, const uint32_t* a, uint32_t bi) {
    asm("add.cc.u32 %0, %0, %2;\n\t"
        "madc.lo.cc.u32 %1, %9, %13, %3;\n\t"
        "madc.hi.cc.u32 %2, %9, %13, %4;\n\t"
        "madc.lo.cc.u32 %3, %10, %13, %5;\n\t"
        "madc.hi.cc.u32 %4, %10, %13, %6;\n\t"
        "madc.lo.cc.u32 %5, %11, %13, %7;\n\t"
        "madc.hi.cc.u32 %6, %11, %13, %8;\n\t"
        "madc.lo.cc.u32 %7, %12, %13, 0;\n\t"
        "madc.hi.u32 %8, %12, %13, 0;"
        : "+r"(even[0]), "+r"(odd[0]), "+r"(odd[1]), "+r"(odd[2]), "+r"(odd[3]), "+r"(odd[4]), "+r"(odd[5]),
          "+r"(odd[6]), "+r"(odd[7])
        : "r"(a[0]), "r"(a[2]), "r"(a[4]), "r"(a[6]), "r"(bi));
  }
  // acc += a[0,2,4,6] * bi (one chain over four pairs), carry-out into top (a fresh hi word)
  static VDF_D void cmad_top(uint32_t* acc, const uint32_t* a, uint32_t bi, uint32_t& top) {
    asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t"
        "madc.hi.cc.u32 %1, %9, %13, %1;\n\t"
        "madc.lo.cc.u32 %2, %10, %13, %2;\n\t"
        "madc.hi.cc.u32 %3, %10, %13, %3;\n\t"
        "madc.lo.cc.u32 %4, %11, %13, %4;\n\t"
        "madc.hi.cc.u32 %5, %11, %13, %5;\n\t"
        "madc.lo.cc.u32 %6, %12, %13, %6;\n\t"
        "madc.hi.cc.u32 %7, %12, %13, %7;\n\t"
        "addc.u32 %8, %8, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]),
          "+r"(acc[7]), "+r"(top)
        : "r"(a[0]), "r"(a[2]), "r"(a[4]), "r"(a[6]), "r"(bi));
  }
  // one Montgomery reduction row specialised to [1, M1, M2, M3, 0, 0, 0, 2^30]; q = -even[0]
  static VDF_D void redc_row(uint32_t* even, uint32_t* odd) {
    uint32_t mi = 0u - even[0];
    const uint32_t M1 = VDF_KMOD[T::ID][0], M2 = VDF_KMOD[T::ID][1], M3 = VDF_KMOD[T::ID][2];
    // odd += q * [M1, M3, 0, 2^30] (pairs at odd columns)
    asm("mad.lo.cc.u32 %0, %8, %9, %0;\n\t"
        "madc.hi.cc.u32 %1, %8, %9, %1;\n\t"
        "madc.lo.cc.u32 %2, %8, %10, %2;\n\t"
        "madc.hi.cc.u32 %3, %8, %10, %3;\n\t"
        "addc.cc.u32 %4, %4, 0;\n\t"
        "addc.cc.u32 %5, %5, 0;\n\t"
        "madc.lo.cc.u32 %6, %8, %11, %6;\n\t"
        "madc.hi.u32 %7, %8, %11, %7;"
        : "+r"(odd[0]), "+r"(odd[1]), "+r"(odd[2]), "+r"(odd[3]), "+r"(odd[4]), "+r"(odd[5]), "+r"(odd[6]),
          "+r"(odd[7])
        : "r"(mi), "r"(M1), "r"(M3), "r"(M7));
    // even += q * [1, M2, 0, 0]; even[0] becomes 0; carry-out into odd[7]
    asm("add.cc.u32 %0, %0, %9;\n\t"
        "addc.cc.u32 %1, %1, 0;\n\t"
        "madc.lo.cc.u32 %2, %9, %10, %2;\n\t"
        "madc.hi.cc.u32 %3, %9, %10, %3;\n\t"
        "addc.cc.u32 %4, %4, 0;\n\t"
        "addc.cc.u32 %5, %5, 0;\n\t"
        "addc.cc.u32 %6, %6, 0;\n\t"
        "addc.cc.u32 %7, %7, 0;\n\t"
        "addc.u32 %8, %8, 0;"
        : "+r"(even[0]), "+r"(even[1]), "+r"(even[2]), "+r"(even[3]), "+r"(even[4]), "+r"(even[5]),
          "+r"(even[6]), "+r"(even[7]), "+r"(odd[7])
        : "r"(mi), "r"(M2));
  }
  static VDF_D void mad_row(uint32_t* even, uint32_t* odd, const uint32_t* a, uint32_t bi, bool first) {
    if (first) {
      mul_n(odd, a + 1, bi);
      mul_n(even, a, bi);
    } else {
      shift_mad(even, odd, a + 1, bi);
      cmad_top(even, a, bi, odd[7]);
    }
    redc_row(even, odd);
  }
  // r = a + b (8 limbs), returns nothing: caller guarantees no carry out
  static VDF_D void add8(uint32_t* r, const uint32_t* a, const uint32_t* b) {
    asm("add.cc.u32 %0, %8, %16;\n\t"
        "addc.cc.u32 %1, %9, %17;\n\t"
        "addc.cc.u32 %2, %10, %18;\n\t"
        "addc.cc.u32 %3, %11, %19;\n\t"
        "addc.cc.u32 %4, %12, %20;\n\t"
        "addc.cc.u32 %5, %13, %21;\n\t"
        "addc.cc.u32 %6, %14, %22;\n\t"
        "addc.u32 %7, %15, %23;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
          "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
  }
  // r = a - b (8 limbs); returns 0xffffffff on borrow, else 0
  static VDF_D uint32_t sub8(uint32_t* r, const uint32_t* a, const uint32_t* b) {
    uint32_t borrow;
    asm("sub.cc.u32 %0, %9, %17;\n\t"
        "subc.cc.u32 %1, %10, %18;\n\t"
        "subc.cc.u32 %2, %11, %19;\n\t"
        "subc.cc.u32 %3, %12, %20;\n\t"
        "subc.cc.u32 %4, %13, %21;\n\t"
        "subc.cc.u32 %5, %14, %22;\n\t"
        "subc.cc.u32 %6, %15, %23;\n\t"
        "subc.cc.u32 %7, %16, %24;\n\t"
        "subc.u32 %8, 0, 0;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(borrow)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
          "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
    return borrow;
  }
  // r = a - m; returns 0xffffffff on borrow (a < m)
  static VDF_D uint32_t sub8_mod(uint32_t* r, const uint32_t* a) {
    uint32_t borrow;
    asm("sub.cc.u32 %0, %9, 1;\n\t"
        "subc.cc.u32 %1, %10, %17;\n\t"
        "subc.cc.u32 %2, %11, %18;\n\t"
        "subc.cc.u32 %3, %12, %19;\n\t"
        "subc.cc.u32 %4, %13, 0;\n\t"
        "subc.cc.u32 %5, %14, 0;\n\t"
        "subc.cc.u32 %6, %15, 0;\n\t"
        "subc.cc.u32 %7, %16, %20;\n\t"
        "subc.u32 %8, 0, 0;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(borrow)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
          "r"(M1), "r"(M2), "r"(M3), "r"(M7));
    return borrow;
  }
  // r = a + m (mod 2^256)
  static VDF_D void add8_mod(uint32_t* r, const uint32_t* a) {
    asm("add.cc.u32 %0, %8, 1;\n\t"
        "addc.cc.u32 %1, %9, %16;\n\t"
        "addc.cc.u32 %2, %10, %17;\n\t"
        "addc.cc.u32 %3, %11, %18;\n\t"
        "addc.cc.u32 %4, %12, 0;\n\t"
        "addc.cc.u32 %5, %13, 0;\n\t"
        "addc.cc.u32 %6, %14, 0;\n\t"
        "addc.u32 %7, %15, %19;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
          "r"(M1), "r"(M2), "r"(M3), "r"(M7));
  }
  // merge the two column sets (even += odd >> 32) and bring the result into [0, m)
  static VDF_D void merge_final(fe& r, uint32_t* even, const uint32_t* odd) {
    asm("add.cc.u32 %0, %0, %8;\n\t"
        "addc.cc.u32 %1, %1, %9;\n\t"
        "addc.cc.u32 %2, %2, %10;\n\t"
        "addc.cc.u32 %3, %3, %11;\n\t"
        "addc.cc.u32 %4, %4, %12;\n\t"
        "addc.cc.u32 %5, %5, %13;\n\t"
        "addc.cc.u32 %6, %6, %14;\n\t"
        "addc.u32 %7, %7, 0;"
        : "+r"(even[0]), "+r"(even[1]), "+r"(even[2]), "+r"(even[3]), "+r"(even[4]), "+r"(even[5]),
          "+r"(even[6]), "+r"(even[7])
        : "r"(odd[1]), "r"(odd[2]), "r"(odd[3]), "r"(odd[4]), "r"(odd[5]), "r"(odd[6]), "r"(odd[7]));
    uint32_t t[8];
    uint32_t borrow = sub8_mod(t, even);
#pragma unroll
    for (int j = 0; j < 8; j++) r.v[j] = borrow ? even[j] : t[j];
  }
  // ---- dedicated squaring ---------------------------------------------------------------------
  // a^2 = sum_i a_i 2^(32 i) * V_i with V_i = a_i 2^(32 i) + 2 * sum_(j>i) a_j 2^(32 j): row i of the multiplication
  // above with the multiplicand V_i = [0 (j < i), a_i, (2a)_(i+1) & ~1, (2a)_(i+2), ...] and the products of its zero
  // limbs dropped -- 36 instead of 64 products, same interleaved reduction, no separate doubling pass (2a < 2^256).
  // tools/ptx_model.py replays these chains carry-exactly against big integers (tests/test_ptx_model.py).
  // shift_mad with the products of the ZO lowest odd limbs (all zero) replaced by carry propagation
  template <int ZO>
  static VDF_D void shift_mad_z(uint32_t* even, uint32_t* odd, const uint32_t* a, uint32_t bi) {
    if constexpr (ZO == 0) {
      shift_mad(even, odd, a, bi);
    } else if constexpr (ZO == 1) {
      asm("add.cc.u32 %0, %0, %2;\n\t"
          "addc.cc.u32 %1, %3, 0;\n\t"
          "addc.cc.u32 %2, %4, 0;\n\t"
          "madc.lo.cc.u32 %3, %9, %12, %5;\n\t"
          "madc.hi.cc.u32 %4, %9, %12, %6;\n\t"
          "madc.lo.cc.u32 %5, %10, %12, %7;\n\t"
          "madc.hi.cc.u32 %6, %10, %12, %8;\n\t"
          "madc.lo.cc.u32 %7, %11, %12, 0;\n\t"
          "madc.hi.u32 %8, %11, %12, 0;"
          : "+r"(even[0]), "+r"(odd[0]), "+r"(odd[1]), "+r"(odd[2]), "+r"(odd[3]), "+r"(odd[4]), "+r"(odd[5]),
            "+r"(odd[6]), "+r"(odd[7])
          : "r"(a[2]), "r"(a[4]), "r"(a[6]), "r"(bi));
    } else if constexpr (ZO == 2) {
      asm("add.cc.u32 %0, %0, %2;\n\t"
          "addc.cc.u32 %1, %3, 0;\n\t"
          "addc.cc.u32 %2, %4, 0;\n\t"
          "addc.cc.u32 %3, %5, 0;\n\t"
          "addc.cc.u32 %4, %6, 0;\n\t"
          "madc.lo.cc.u32 %5, %9, %11, %7;\n\t"
          "madc.hi.cc.u32 %6, %9, %11, %8;\n\t"
          "madc.lo.cc.u32 %7, %10, %11, 0;\n\t"
          "madc.hi.u32 %8, %10, %11, 0;"
          : "+r"(even[0]), "+r"(odd[0]), "+r"(odd[1]), "+r"(odd[2]), "+r"(odd[3]), "+r"(odd[4]), "+r"(odd[5]),
            "+r"(odd[6]), "+r"(odd[7])
          : "r"(a[4]), "r"(a[6]), "r"(bi));
    } else {
      static_assert(ZO == 3, "at most three zero odd limbs");
      asm("add.cc.u32 %0, %0, %2;\n\t"
          "addc.cc.u32 %1, %3, 0;\n\t"
          "addc.cc.u32 %2, %4, 0;\n\t"
          "addc.cc.u32 %3, %5, 0;\n\t"
          "addc.cc.u32 %4, %6, 0;\n\t"
          "addc.cc.u32 %5, %7, 0;\n\t"
          "addc.cc.u32 %6, %8, 0;\n\t"
          "madc.lo.cc.u32 %7, %9, %10, 0;\n\t"
          "madc.hi.u32 %8, %9, %10, 0;"
          : "+r"(even[0]), "+r"(odd[0]), "+r"(odd[1]), "+r"(odd[2]), "+r"(odd[3]), "+r"(odd[4]), "+r"(odd[5]),
            "+r"(odd[6]), "+r"(odd[7])
          : "r"(a[6]), "r"(bi));
    }
  }
  // cmad_top starting at the first non-zero even limb (ZE leading zero limbs add nothing and carry nothing)
  template <int ZE>
  static VDF_D void cmad_top_z(uint32_t* acc, const uint32_t* a, uint32_t bi, uint32_t& top) {
    if constexpr (ZE == 0) {
      cmad_top(acc, a, bi, top);
    } else if constexpr (ZE == 1) {
      asm("mad.lo.cc.u32 %0, %7, %10, %0;\n\t"
          "madc.hi.cc.u32 %1, %7, %10, %1;\n\t"
          "madc.lo.cc.u32 %2, %8, %10, %2;\n\t"
          "madc.hi.cc.u32 %3, %8, %10, %3;\n\t"
          "madc.lo.cc.u32 %4, %9, %10, %4;\n\t"
          "madc.hi.cc.u32 %5, %9, %10, %5;\n\t"
          "addc.u32 %6, %6, 0;"
          : "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "+r"(top)
          : "r"(a[2]), "r"(a[4]), "r"(a[6]), "r"(bi));
    } else if constexpr (ZE == 2) {
      asm("mad.lo.cc.u32 %0, %5, %7, %0;\n\t"
          "madc.hi.cc.u32 %1, %5, %7, %1;\n\t"
          "madc.lo.cc.u32 %2, %6, %7, %2;\n\t"
          "madc.hi.cc.u32 %3, %6, %7, %3;\n\t"
          "addc.u32 %4, %4, 0;"
          : "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "+r"(top)
          : "r"(a[4]), "r"(a[6]), "r"(bi));
    } else if constexpr (ZE == 3) {
      asm("mad.lo.cc.u32 %0, %3, %4, %0;\n\t"
          "madc.hi.cc.u32 %1, %3, %4, %1;\n\t"
          "addc.u32 %2, %2, 0;"
          : "+r"(acc[6]), "+r"(acc[7]), "+r"(top)
          : "r"(a[6]), "r"(bi));
    } else {
      static_assert(ZE == 4, "at most four zero even limbs");
    }
  }
  // row I of the squaring: first/second play even/odd as in mad_row
  template <int I>
  static VDF_D void sqr_row(uint32_t* first, uint32_t* second, const uint32_t* a, const uint32_t* d) {
    uint32_t v[8];
#pragma unroll
    for (int j = 0; j < 8; j++) v[j] = j < I ? 0u : (j == I ? a[j] : (j == I + 1 ? (d[j] & 0xfffffffeu) : d[j]));
    if constexpr (I == 0) {
      mul_n(second, v + 1, a[0]);
      mul_n(first, v, a[0]);
    } else {
      shift_mad_z<I / 2>(first, second, v + 1, a[I]);
      cmad_top_z<(I + 1) / 2>(first, v, a[I], second[7]);
    }
    redc_row(first, second);
  }
#endif

  static VDF_HD fe mul(const fe& a, const fe& b) {
    fe r;
#if defined(__CUDA_ARCH__)
    uint32_t even[8], odd[8];
#pragma unroll
    for (int i = 0; i < 8; i += 2) {
      mad_row(even, odd, a.v, b.v[i], i == 0);
      mad_row(odd, even, a.v, b.v[i + 1], false);
    }
    merge_final(r, even, odd);
#else
    // CIOS over 4 x 64-bit limbs: the 32-bit limbs above read as little-endian u64 pairs, m = [(M1 << 32) | 1,
    // (M3 << 32) | M2, 0, 2^62] and -m^-1 mod 2^64 = (M1 << 32) - 1
    typedef unsigned __int128 u128;
    const uint64_t m[4] = {((uint64_t)M1 << 32) | 1u, ((uint64_t)M3 << 32) | M2, 0, (uint64_t)M7 << 32};
    const uint64_t minv = ((uint64_t)M1 << 32) - 1u;
    uint64_t x[4], y[4], t[6] = {0, 0, 0, 0, 0, 0};
    std::memcpy(x, a.v, 32);
    std::memcpy(y, b.v, 32);
    for (int i = 0; i < 4; i++) {
      u128 c = 0;
      for (int j = 0; j < 4; j++) {
        c += (u128)x[j] * y[i] + t[j];
        t[j] = (uint64_t)c;
        c >>= 64;
      }
      c += t[4];
      t[4] = (uint64_t)c;
      t[5] = (uint64_t)(c >> 64);
      const uint64_t q = t[0] * minv;
      c = ((u128)q * m[0] + t[0]) >> 64;
      for (int j = 1; j < 4; j++) {
        c += (u128)q * m[j] + t[j];
        t[j - 1] = (uint64_t)c;
        c >>= 64;
      }
      c += t[4];
      t[3] = (uint64_t)c;
      t[4] = t[5] + (uint64_t)(c >> 64);
    }
    uint64_t s[4];
    u128 bw = 0;
    for (int j = 0; j < 4; j++) {
      const u128 d = (u128)t[j] - m[j] - (uint64_t)bw;
      s[j] = (uint64_t)d;
      bw = (d >> 64) & 1;
    }
    const bool ge = t[4] != 0 || bw == 0;
    for (int j = 0; j < 4; j++) t[j] = ge ? s[j] : t[j];
    std::memcpy(r.v, t, 32);
#endif
    return r;
  }

  static VDF_HD fe sqr(const fe& a) {
#if defined(__CUDA_ARCH__)
    fe r;
    uint32_t d[8], even[8], odd[8];
    add8(d, a.v, a.v);   // 2a < 2^256 (a < m < 2^255)
    sqr_row<0>(even, odd, a.v, d);
    sqr_row<1>(odd, even, a.v, d);
    sqr_row<2>(even, odd, a.v, d);
    sqr_row<3>(odd, even, a.v, d);
    sqr_row<4>(even, odd, a.v, d);
    sqr_row<5>(odd, even, a.v, d);
    sqr_row<6>(even, odd, a.v, d);
    sqr_row<7>(odd, even, a.v, d);
    merge_final(r, even, odd);
    return r;
#else
    return mul(a, a);
#endif
  }

  // Out-of-line copy for kernels whose fully inlined body would overflow the instruction cache (the bucket
  // accumulation inlines ~20 multiplications): one shared 250-instruction body instead.
#if defined(__CUDACC__)
  static __device__ __noinline__ fe mul_call(const fe& a, const fe& b) { return mul(a, b); }
  static __device__ __noinline__ fe sqr_call(const fe& a) { return sqr(a); }
  // operands and result in registers (by value): no trip through the local-memory stack around the call
  static __device__ __noinline__ fe mul_val(fe a, fe b) { return mul(a, b); }
  static __device__ __noinline__ fe sqr_val(fe a) { return sqr(a); }
#else
  static fe mul_val(fe a, fe b) { return mul(a, b); }
  static fe sqr_val(fe a) { return sqr(a); }
  static fe mul_call(const fe& a, const fe& b) { return mul(a, b); }
  static fe sqr_call(const fe& a) { return sqr(a); }
#endif

  // Montgomery -> canonical: multiply by the integer 1
  static VDF_HD fe from_mont(const fe& a) {
    fe o = zero();
    o.v[0] = 1;
    return mul(a, o);
  }

  // a^(m-2) (Fermat); m - 2 has limbs [0xffffffff, M1-1, M2, M3, 0, 0, 0, 2^30].  Cold paths only
  // (normalising one result point), so a plain square-and-multiply loop, not unrolled.
  static VDF_HD fe inv(const fe& a) {
    fe r = one();
#pragma unroll 1
    for (int j = 7; j >= 0; j--) {
      uint32_t e = j == 0 ? 0xffffffffu : j == 1 ? M1 - 1u : mod_limb(j);
#pragma unroll 1
      for (int bit = 31; bit >= 0; bit--) {
        r = sqr(r);
        if ((e >> bit) & 1u) r = mul(r, a);
      }
    }
    return r;
  }
};

typedef Field<FpTag> Fp;
typedef Field<FqTag> Fq;

// ---- 32-byte vector load/store (two 128-bit transactions) ----------------------------------------
VDF_HD fe fe_load(const void* p) {
  fe r;
#if defined(__CUDA_ARCH__)
  const uint4* q = reinterpret_cast<const uint4*>(p);
  uint4 a = q[0], b = q[1];
  r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w;
  r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
#else
  const uint32_t* q = reinterpret_cast<const uint32_t*>(p);
  for (int j = 0; j < 8; j++) r.v[j] = q[j];
#endif
  return r;
}

// Load for RANDOM 32 / 64-byte gathers (points picked by the sorted references): read-only path and the smallest
// L2 prefetch size, so that a miss does not pull the neighbouring sectors of the 128-byte line from DRAM.
#ifndef VDF_GATHER_L2
#define VDF_GATHER_L2 64
#endif
VDF_HD fe fe_load_gather(const void* p) {
#if defined(__CUDA_ARCH__) && VDF_GATHER_L2 > 0
  fe r;
#define VDF_STR2(x) #x
#define VDF_STR(x) VDF_STR2(x)
  asm volatile("ld.global.nc.L2::" VDF_STR(VDF_GATHER_L2) "B.v4.u32 {%0,%1,%2,%3}, [%8];\n\t"
               "ld.global.nc.L2::" VDF_STR(VDF_GATHER_L2) "B.v4.u32 {%4,%5,%6,%7}, [%8+16];"
               : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]),
                 "=r"(r.v[7])
               : "l"(p));
#undef VDF_STR
#undef VDF_STR2
  return r;
#else
  return fe_load(p);
#endif
}

VDF_HD void fe_store(void* p, const fe& a) {
#if defined(__CUDA_ARCH__)
  uint4* q = reinterpret_cast<uint4*>(p);
  q[0] = make_uint4(a.v[0], a.v[1], a.v[2], a.v[3]);
  q[1] = make_uint4(a.v[4], a.v[5], a.v[6], a.v[7]);
#else
  uint32_t* q = reinterpret_cast<uint32_t*>(p);
  for (int j = 0; j < 8; j++) q[j] = a.v[j];
#endif
}

}  // namespace vdf
