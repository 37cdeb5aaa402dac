// tests/emul: the Spartan prover's functors (r1cs.cuh PaddedLayout, OuterTablesFn, PaddedScatterFn; sumcheck.cuh
// MultiDot, IpaJoinFn) run by a CPU loop through vdf::HostLaunch, for `pytest -m "not gpu"` (tests/test_spartan.py).
// TEST TOOL ONLY, like emul.cpp: libvdfgpu.so never contains this code.  All elements are 32-byte Montgomery; field
// 0 = Fp, 1 = Fq; the shape is the library's stacked CSR (3 cons rows: A, then B, then C).
#include <cstdint>
#include <cstring>

#include "../../vdf_b200/csrc/r1cs.cuh"
#include "../../vdf_b200/csrc/sumcheck.cuh"

using namespace vdf;

template <class F>
static void outer_tables(const uint32_t* row_ptr, const uint32_t* col, const void* val, uint32_t cons, uint32_t vars,
                         uint32_t io, const void* W, const void* uX, const void* E, size_t m, void* out4) {
  const fe* ux = (const fe*)uX;
  fe* o = (fe*)out4;
  HostLaunch L;
  L.run(m, OuterTablesFn<F>{CsrView{row_ptr, col, (const fe*)val, cons, vars, io}, ZView{(const fe*)W, ux, ux + 1},
                            (const fe*)E, o, o + m, o + 2 * m, o + 3 * m});
}

template <class F>
static void scatter(uint32_t cons, uint32_t vars, uint32_t io, const void* M, const void* W, const void* uX, void* Mp,
                    void* zp) {
  const PaddedLayout pad = PaddedLayout::of(cons, vars, io);
  const fe* ux = (const fe*)uX;
  HostLaunch L;
  L.run(2 * pad.m, PaddedScatterFn<F>{pad, (const fe*)M, ZView{(const fe*)W, ux, ux + 1}, (fe*)Mp, (fe*)zp});
}

template <class F>
static void multi_dot3(const void* const* v, const void* const* eq, const size_t* len, size_t n, void* out3) {
  MultiDot<3> d;
  for (int q = 0; q < 3; q++) {
    d.v[q] = (const fe*)v[q];
    d.eq[q] = (const fe*)eq[q];
    d.len[q] = len[q];
  }
  fe acc[3] = {F::zero(), F::zero(), F::zero()};
  for (size_t i = 0; i < n; i++) d.template add_terms<F>(acc, i);   // the kernel's per-thread loop, one thread
  std::memcpy(out3, acc, sizeof(acc));
}

template <class F>
static void ipa_join(const void* E, const void* W, const void* eqx, const void* eqy, const void* rho, size_t n, void* a,
                     void* b) {
  fe r;
  std::memcpy(&r, rho, sizeof(fe));
  HostLaunch L;
  L.run(n, IpaJoinFn<F>{(const fe*)E, (const fe*)W, (const fe*)eqx, (const fe*)eqy, r, (fe*)a, (fe*)b});
}

extern "C" {

// m, whether 1 + io fits, and the padded column of each shape column c < vars + 1 + io (out_cols), and the source
// column of each padded index j < 2m (-1: padding) (out_src)
uint64_t emul_padded_layout(uint32_t cons, uint32_t vars, uint32_t io, int* fits, uint64_t* out_cols, int64_t* out_src) {
  const PaddedLayout pad = PaddedLayout::of(cons, vars, io);
  *fits = pad.fits();
  for (uint32_t c = 0; c < vars + 1 + io; c++) out_cols[c] = pad.col(c);
  for (size_t j = 0; j < 2 * pad.m; j++) out_src[j] = pad.source(j);
  return pad.m;
}

// out4: Az, Bz, Cz, D, m elements each
void emul_outer_tables(int field, const uint32_t* row_ptr, const uint32_t* col, const void* val, uint32_t cons,
                       uint32_t vars, uint32_t io, const void* W, const void* uX, const void* E, size_t m, void* out4) {
  if (field == 0) outer_tables<Fp>(row_ptr, col, val, cons, vars, io, W, uX, E, m, out4);
  else outer_tables<Fq>(row_ptr, col, val, cons, vars, io, W, uX, E, m, out4);
}

// Mp, zp: 2m elements each; M: vars + 1 + io elements
void emul_padded_scatter(int field, uint32_t cons, uint32_t vars, uint32_t io, const void* M, const void* W,
                         const void* uX, void* Mp, void* zp) {
  if (field == 0) scatter<Fp>(cons, vars, io, M, W, uX, Mp, zp);
  else scatter<Fq>(cons, vars, io, M, W, uX, Mp, zp);
}

void emul_multi_dot3(int field, const void* const* v, const void* const* eq, const size_t* len, size_t n, void* out3) {
  if (field == 0) multi_dot3<Fp>(v, eq, len, n, out3);
  else multi_dot3<Fq>(v, eq, len, n, out3);
}

void emul_ipa_join(int field, const void* E, const void* W, const void* eqx, const void* eqy, const void* rho, size_t n,
                   void* a, void* b) {
  if (field == 0) ipa_join<Fp>(E, W, eqx, eqy, rho, n, a, b);
  else ipa_join<Fq>(E, W, eqx, eqy, rho, n, a, b);
}

}  // extern "C"
