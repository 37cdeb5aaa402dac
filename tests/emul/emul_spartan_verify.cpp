// tests/emul: the batched sparse evaluation of the Spartan verifier (r1cs.cuh EqHalves, EqHalfTablesBatchFn,
// SparseEvalBatchFn) run by a CPU loop through vdf::HostLaunch, for `pytest -m "not gpu"` (tests/test_spartan_verify.py).
// TEST TOOL ONLY, like emul.cpp: libvdfgpu.so never contains this code.  All elements are 32-byte Montgomery; field
// 0 = Fp, 1 = Fq; the shape is the library's stacked CSR (3 cons rows: A, then B, then C).
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../vdf_b200/csrc/r1cs.cuh"

using namespace vdf;

template <class F>
static void half_tables(size_t k, uint32_t ell_x, const void* rx, const void* ry, void* out) {
  HostLaunch L;
  const EqHalves h = EqHalves::of(ell_x);
  L.run(k * h.per, EqHalfTablesBatchFn<F>{(const fe*)rx, (const fe*)ry, ell_x, h, (fe*)out});
}

// the kernel's per-thread loop with the proof fixed, one thread per proof over every row
template <class F>
static void sparse_eval(const uint32_t* row_ptr, const uint32_t* col, const void* val, uint32_t cons, uint32_t vars,
                        uint32_t io, size_t k, const void* rx, const void* ry, void* out3) {
  const PaddedLayout pad = PaddedLayout::of(cons, vars, io);
  const EqHalves h = EqHalves::of(pad.ell_x);
  std::vector<fe> tables(k * h.per);
  HostLaunch L;
  L.run(k * h.per, EqHalfTablesBatchFn<F>{(const fe*)rx, (const fe*)ry, pad.ell_x, h, tables.data()});
  const SparseEvalBatchFn<F> f{CsrView{row_ptr, col, (const fe*)val, cons, vars, io}, pad, h, tables.data(), k};
  fe* o = (fe*)out3;
  for (size_t q = 0; q < k; q++) {
    fe acc[3] = {F::zero(), F::zero(), F::zero()};
    for (uint32_t row = 0; row < cons; row++) f.add_row(acc, q, row);
    std::memcpy(o + 3 * q, acc, sizeof(acc));
  }
}

extern "C" {

// entries per proof of the half tables at ell_x, and each table's size in bits (bits4)
uint64_t emul_eq_halves(uint32_t ell_x, uint32_t* bits4) {
  const EqHalves h = EqHalves::of(ell_x);
  for (int t = 0; t < 4; t++) bits4[t] = h.bits[t];
  return h.per;
}

// out: [k][per] Hi(r_x), Lo(r_x), Hi(r_y), Lo(r_y)
void emul_eq_half_tables(int field, size_t k, uint32_t ell_x, const void* rx, const void* ry, void* out) {
  if (field == 0) half_tables<Fp>(k, ell_x, rx, ry, out);
  else half_tables<Fq>(k, ell_x, rx, ry, out);
}

// out3: [k][3] = (A, B, C)(r_x[q], r_y[q]); rx: [k][ell_x], ry: [k][ell_x + 1]
void emul_sparse_eval_batch(int field, const uint32_t* row_ptr, const uint32_t* col, const void* val, uint32_t cons,
                            uint32_t vars, uint32_t io, size_t k, const void* rx, const void* ry, void* out3) {
  if (field == 0) sparse_eval<Fp>(row_ptr, col, val, cons, vars, io, k, rx, ry, out3);
  else sparse_eval<Fq>(row_ptr, col, val, cons, vars, io, k, rx, ry, out3);
}

}  // extern "C"
