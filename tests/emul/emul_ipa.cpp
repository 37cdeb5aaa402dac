// tests/emul: the inner-product argument's expansion and fold functors (sumcheck.cuh IpaExpandFn, IpaFoldFn) run by
// a CPU loop through vdf::HostLaunch, for `pytest -m "not gpu"` (tests/test_ipa.py).  TEST TOOL ONLY, like emul.cpp:
// libvdfgpu.so never contains this code.  All elements are 32-byte Montgomery; field 0 = Fp, 1 = Fq.
#include <cstdint>
#include <cstring>

#include "../../vdf_b200/csrc/sumcheck.cuh"

using namespace vdf;

template <class F>
static void expand(const void* a, const void* coef, const void* c2, const void* u_scale, uint32_t log_m, size_t n,
                   void* SL, void* SR) {
  fe u;
  std::memcpy(&u, u_scale, sizeof(fe));
  HostLaunch L;
  L.run(n + 1, IpaExpandFn<F>{(const fe*)a, (const fe*)coef, (const fe*)c2, u, log_m, n, (fe*)SL, (fe*)SR});
}

template <class F>
static void fold(void* a, void* b, size_t h, const void* coef_in, void* coef_out, size_t nc, const void* r,
                 const void* r_inv) {
  fe rv, ri;
  std::memcpy(&rv, r, sizeof(fe));
  std::memcpy(&ri, r_inv, sizeof(fe));
  HostLaunch L;
  L.run(h > nc ? h : nc, IpaFoldFn<F>{(fe*)a, (fe*)b, h, (const fe*)coef_in, (fe*)coef_out, nc, rv, ri});
}

extern "C" {

// SL, SR: n + 1 elements each; a: 2^log_m elements; coef: n / 2^log_m elements; c2 = (c_L, c_R)
void emul_ipa_expand(int field, const void* a, const void* coef, const void* c2, const void* u_scale, uint32_t log_m,
                     size_t n, void* SL, void* SR) {
  if (field == 0) expand<Fp>(a, coef, c2, u_scale, log_m, n, SL, SR);
  else expand<Fq>(a, coef, c2, u_scale, log_m, n, SL, SR);
}

// a, b: 2h elements, halved in place; coef_out[2t + beta] from coef_in[t], t < nc; a and b may be NULL when h = 0
void emul_ipa_fold(int field, void* a, void* b, size_t h, const void* coef_in, void* coef_out, size_t nc, const void* r,
                   const void* r_inv) {
  if (field == 0) fold<Fp>(a, b, h, coef_in, coef_out, nc, r, r_inv);
  else fold<Fq>(a, b, h, coef_in, coef_out, nc, r, r_inv);
}

}  // extern "C"
