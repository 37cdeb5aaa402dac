// tests/emul: the scalar table of batched inner-product verification (sumcheck.cuh IpaHalfTablesFn,
// IpaBatchScalarsFn) run by a CPU loop through vdf::HostLaunch, for `pytest -m "not gpu"` (tests/test_ipa_verify.py).
// TEST TOOL ONLY, like emul.cpp: libvdfgpu.so never contains this code.  All elements are 32-byte Montgomery; field
// 0 = Fp, 1 = Fq.
#include <cstdint>
#include <cstring>

#include "../../vdf_b200/csrc/sumcheck.cuh"

using namespace vdf;

template <class F>
static void half_tables(const void* r, const void* r_inv, const void* scale, uint32_t ell, uint32_t lo_bits, size_t k,
                        void* hi, void* lo) {
  HostLaunch L;
  L.run(k * (((size_t)1 << (ell - lo_bits)) + ((size_t)1 << lo_bits)),
        IpaHalfTablesFn<F>{(const fe*)r, (const fe*)r_inv, (const fe*)scale, ell, lo_bits, k, (fe*)hi, (fe*)lo});
}

template <class F>
static void batch_scalars(const void* hi, const void* lo, uint32_t hi_bits, uint32_t lo_bits, size_t k,
                          const void* last, void* S) {
  fe l;
  std::memcpy(&l, last, sizeof(fe));
  HostLaunch L;
  L.run(((size_t)1 << (hi_bits + lo_bits)) + 1,
        IpaBatchScalarsFn<F>{(const fe*)hi, (const fe*)lo, hi_bits, lo_bits, k, l, (fe*)S});
}

extern "C" {

// r, r_inv: [k][ell]; scale: [k]; hi: [k][2^(ell - lo_bits)]; lo: [k][2^lo_bits]
void emul_ipa_half_tables(int field, const void* r, const void* r_inv, const void* scale, uint32_t ell,
                          uint32_t lo_bits, size_t k, void* hi, void* lo) {
  if (field == 0) half_tables<Fp>(r, r_inv, scale, ell, lo_bits, k, hi, lo);
  else half_tables<Fq>(r, r_inv, scale, ell, lo_bits, k, hi, lo);
}

// S: 2^(hi_bits + lo_bits) + 1 elements, the last one = *last
void emul_ipa_batch_scalars(int field, const void* hi, const void* lo, uint32_t hi_bits, uint32_t lo_bits, size_t k,
                            const void* last, void* S) {
  if (field == 0) batch_scalars<Fp>(hi, lo, hi_bits, lo_bits, k, last, S);
  else batch_scalars<Fq>(hi, lo, hi_bits, lo_bits, k, last, S);
}

}  // extern "C"
