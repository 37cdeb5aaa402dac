// tests/emul: the satisfiability functor (r1cs.cuh: SatInitFn + RelaxedSatFn) run by a CPU loop through
// vdf::HostLaunch, for `pytest -m "not gpu"` (tests/test_r1cs_sat.py).  TEST TOOL ONLY, like emul.cpp: libvdfgpu.so
// never contains this code.  The host path of the functor counts with plain additions and a plain minimum; the
// warp-ballot path is the GPU's and is checked on the device (tests/test_gpu_r1cs_sat.py).
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../vdf_b200/csrc/r1cs.cuh"
#include "../../vdf_b200/csrc/r1cs_host.hpp"

using namespace vdf;

extern "C" {

// counts2_out[0] = rows with Az.Bz != u.Cz + E, counts2_out[1] = the smallest such row (num_cons when none).
// E NULL means E = 0; z = [W | u | X].  Returns -1 when the COO input is malformed.
int emul_r1cs_sat(int field, size_t num_cons, size_t num_vars, size_t num_io, const uint64_t* a_rows,
                  const uint64_t* a_cols, const void* a_vals, size_t a_nnz, const uint64_t* b_rows, const uint64_t* b_cols,
                  const void* b_vals, size_t b_nnz, const uint64_t* c_rows, const uint64_t* c_cols, const void* c_vals,
                  size_t c_nnz, const void* W, const void* E, const void* u, const void* X, uint64_t* counts2_out) {
  const uint64_t* rows[3] = {a_rows, b_rows, c_rows};
  const uint64_t* cols[3] = {a_cols, b_cols, c_cols};
  const uint8_t* vals[3] = {(const uint8_t*)a_vals, (const uint8_t*)b_vals, (const uint8_t*)c_vals};
  size_t nnzs[3] = {a_nnz, b_nnz, c_nnz};
  HostCsr csr;
  try {
    csr = coo_to_csr(num_cons, num_vars + 1 + num_io, rows, cols, vals, nnzs);
  } catch (const std::exception&) {
    return -1;
  }
  std::vector<fe> val(csr.val.size() / 32 + 1), w(num_vars + 1), e(num_cons), ux(1 + num_io);
  std::memcpy(val.data(), csr.val.data(), csr.val.size());
  std::memcpy(w.data(), W, num_vars * 32);
  if (E) std::memcpy(e.data(), E, num_cons * 32);
  std::memcpy(ux.data(), u, 32);
  std::memcpy(ux.data() + 1, X, num_io * 32);
  CsrView m{csr.row_ptr.data(), csr.col.data(), val.data(), (uint32_t)num_cons, (uint32_t)num_vars, (uint32_t)num_io};
  ZView z{w.data(), ux.data(), ux.data() + 1};
  uint32_t words[4];   // the two little-endian u64 counters as the library's device buffer holds them
  HostLaunch L;
  L.run(1, SatInitFn{words, (uint32_t)num_cons});
  if (field == 0) L.run(num_cons, RelaxedSatFn<Fp>{m, z, E ? e.data() : nullptr, words, words + 2});
  else L.run(num_cons, RelaxedSatFn<Fq>{m, z, E ? e.data() : nullptr, words, words + 2});
  counts2_out[0] = words[0] | (uint64_t)words[1] << 32;
  counts2_out[1] = words[2] | (uint64_t)words[3] << 32;
  return 0;
}

}  // extern "C"
