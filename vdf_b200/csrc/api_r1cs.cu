// C ABI, part 2: R1CS shape upload (COO -> CSR), multiply_vec, commit_T, fold, and the device-resident
// running instance used for a chain of fold steps.  Contract and reference pointers: include/vdfgpu.h.
#include <algorithm>
#include <cstring>
#include <memory>
#include <type_traits>
#include <vector>

#include "ctx.cuh"
#include "minroot.cuh"
#include "r1cs.cuh"
#include "r1cs_host.hpp"
#include "sumcheck.cuh"

struct vdfgpu_r1cs {
  int field = 0;
  uint32_t cons = 0, vars = 0, io = 0;
  size_t nnz = 0;
  uint32_t* row_ptr = nullptr;  // [3*cons+1]
  uint32_t* col = nullptr;
  vdf::fe* val = nullptr;
  uint32_t* col_ptr = nullptr;    // column view (csr_to_csc): [vars + 1 + io + 1]
  uint32_t* csc_row = nullptr;    // [nnz]
  vdf::fe* csc_val = nullptr;     // [nnz]
  uint32_t* heavy = nullptr;      // [n_heavy]
  uint32_t n_heavy = 0;
  mutable int refs = 0;   // running instances and Spartan proofs in progress holding this shape (vdfgpu_r1cs_destroy
                          // refuses while > 0)
  vdf::CsrView view() const { return vdf::CsrView{row_ptr, col, val, cons, vars, io}; }
  vdf::CscView col_view() const { return vdf::CscView{col_ptr, csc_row, csc_val, heavy, vdf::HostCsc::HEAVY}; }
  ~vdfgpu_r1cs() {   // the one release path: failed create, vdfgpu_r1cs_destroy
    cudaFree(row_ptr); cudaFree(col); cudaFree(val);
    cudaFree(col_ptr); cudaFree(csc_row); cudaFree(csc_val); cudaFree(heavy);
  }
};

struct vdfgpu_running {
  const vdfgpu_r1cs* shape = nullptr;
  vdfgpu_gens* gens = nullptr;
  vdf::fe* W = nullptr;   // running witness [vars]
  vdf::fe* E = nullptr;   // running error   [cons]
  vdf::fe* uX = nullptr;  // [1 + io]: u then X
  vdf::fe* W2 = nullptr;  // fresh witness  [vars]
  vdf::fe* uX2 = nullptr; // [1 + io]: 1 then X2
  vdf::fe* T = nullptr;   // cross-term [cons]
  vdf::fe* r = nullptr;   // challenge
  vdf::jac_t* comm = nullptr;  // [2] comm_W2, comm_T
  uint8_t* bounce = nullptr;   // pinned: both commitments come back with one asynchronous copy; [1 + io] staging of uX2 behind it
  // recorded behind the work of every call on this instance, waited on before the next one enqueues: a call on another
  // stream or thread (vdfgpu_running_finish returns before its fold has run) is ordered behind the previous one
  cudaEvent_t done = nullptr;
  bool have_running = false, have_fresh = false;
  int refs = 0;   // Spartan proofs in progress on this instance (vdfgpu_running_destroy refuses while > 0)
  ~vdfgpu_running() {   // the one release path: failed create, vdfgpu_running_destroy
    if (bounce) cudaFreeHost(bounce);
    if (done) cudaEventDestroy(done);
    cudaFree(W); cudaFree(W2); cudaFree(E); cudaFree(T); cudaFree(uX); cudaFree(uX2);
    cudaFree(r); cudaFree(comm);
  }
};

// Step-circuit witnesses of all n steps of one proof, generated on the device (SURVEY 8f rank 1) on a side stream
struct vdfgpu_witness_bank {
  int field = 0;
  uint64_t t = 0;
  size_t n = 0;
  vdf::fe* w = nullptr;         // [n][4t + 1]
  cudaStream_t stream = nullptr;
  cudaEvent_t ready = nullptr;
  ~vdfgpu_witness_bank() {   // the one release path: failed create, vdfgpu_witness_bank_destroy
    if (w) cudaFree(w);
    if (ready) cudaEventDestroy(ready);
    if (stream) cudaStreamDestroy(stream);
  }
};

namespace vdf {

static void launch_multiply_vec(CudaLaunch& L, const vdfgpu_r1cs* s, ZView z, fe* Az, fe* Bz, fe* Cz) {
  with_field(s->field, "r1cs", [&](auto f) {
    L.run<128>(3 * (size_t)s->cons, MultiplyVecFn<decltype(f)>{s->view(), z, Az, Bz, Cz});
  });
}

static void launch_cross_term(CudaLaunch& L, const vdfgpu_r1cs* s, ZView z1, ZView z2, fe* T) {
#ifndef VDF_CT_MINB
#define VDF_CT_MINB 8
#endif
  with_field(s->field, "r1cs", [&](auto f) {
    L.run<128, VDF_CT_MINB>(s->cons, CrossTermFn<decltype(f)>{s->view(), z1, z2, T});
  });
}

template <class F>
static void launch_fold(CudaLaunch& L, fe* W1, const fe* W2, size_t nW, fe* E1, const fe* T, size_t nE, const fe* r) {
  L.run<256>(nW + nE, FoldFn<F>{W1, W2, nW, E1, T, nE, r});
}

// the scalar field of the commitment curve must be the R1CS field
static void check_gens_field(const vdfgpu_r1cs* s, const vdfgpu_gens* g, const std::string& who = "") {
  const bool same = with_curve(g->curve, "gens", [&](auto, auto, auto SF) {
    return with_field(s->field, "r1cs", [](auto f) { return std::is_same<decltype(f), decltype(SF)>::value; });
  });
  if (!same) throw ArgError(who + "generator curve's scalar field differs from the R1CS field");
}

void upload_constants_r1cs() { VDF_CUDA_CHECK(upload_field_constants()); }

static fe host_one(int field) { return with_field(field, "r1cs", [](auto f) { return decltype(f)::one(); }); }

// every vdfgpu_running_* call that enqueues work: running_after() before its first operation on `st`,
// running_done() after its last
static void running_after(const vdfgpu_running* f, cudaStream_t st) { VDF_CUDA_CHECK(cudaStreamWaitEvent(st, f->done, 0)); }
static void running_done(const vdfgpu_running* f, cudaStream_t st) { VDF_CUDA_CHECK(cudaEventRecord(f->done, st)); }

// ---- satisfiability checks (vdfgpu_r1cs_is_sat_relaxed*, vdfgpu_running_check) ----------------------------------
// counts2: the two u64 of the C ABI, as four u32 words on the device (see SatInitFn)
static void launch_sat(CudaLaunch& L, const vdfgpu_r1cs* s, ZView z, const fe* E, uint64_t* counts2) {
  uint32_t* words = reinterpret_cast<uint32_t*>(counts2);
  uint32_t* bad = words;
  uint32_t* first = words + 2;
  L.run<32>(1, SatInitFn{words, s->cons});
  with_field(s->field, "r1cs", [&](auto f) {
    L.run<128, 8>(s->cons, RelaxedSatFn<decltype(f)>{s->view(), z, E, bad, first});
  });
}

// What one check brings back to the host: the two counters and commit(W), commit(E) as un-normalised points, in ONE
// device block [counts2 | pad to 96 B | point | point] copied with one D2H.
struct SatResult {
  uint64_t counts[2] = {0, 0};
  uint8_t comm[2][96] = {};
};
constexpr size_t SAT_BLOCK = 3 * sizeof(jac_t);
static_assert(sizeof(jac_t) == 96, "points are 96 bytes");

// pinned landing zone of the read-back, one per calling thread (the previous call on this thread has been waited for)
static uint8_t* pinned_sat() {
  static thread_local uint8_t* p = nullptr;
  if (!p) VDF_CUDA_CHECK(cudaHostAlloc((void**)&p, SAT_BLOCK, cudaHostAllocDefault));
  return p;
}

static void check_sat_gens(const vdfgpu_r1cs* s, const vdfgpu_gens* g, const char* what) {
  check_gens_field(s, g);
  if (g->n < s->cons || g->n < s->vars) throw ArgError(std::string(what) + ": fewer generators than max(vars, cons)");
}

// Row check, then commit(W) and commit(E) in ONE batched MSM pass (as running_commit_enqueue batches commit(W2) and
// commit(T)), then one D2H into pinned memory; the wait happens after the context lock is released.  The points are
// computed un-normalised whatever the set's flags and normalised on the host once they have landed (`res`).
static void sat_enqueue(const vdfgpu_r1cs* s, vdfgpu_gens* gens, const fe* W, const fe* E, const fe* uX, bool want_W,
                        bool want_E, SatResult& res) {
  cudaStream_t st = cur_stream();
  CudaLaunch L = api_launch(st);
  DevBuf<jac_t> out(3, st);
  launch_sat(L, s, ZView{W, uX, uX + 1}, E, reinterpret_cast<uint64_t*>(out.p));
  const fe* vecs[2];
  size_t lens[2];
  uint32_t k = 0;
  if (want_W) { vecs[k] = W; lens[k++] = s->vars; }
  if (want_E) { vecs[k] = E; lens[k++] = s->cons; }
  if (k) msm_batch_on_device(gens, vecs, lens, k, out.p + 1, true);
  uint8_t* pin = pinned_sat();
  d2h(pin, out.p, 96 + k * sizeof(jac_t), st);
  sync_after_unlock(st);
  copy_after_sync(res.counts, pin, sizeof(res.counts));
  for (uint32_t j = 0, slot = 0; j < 2; j++) {
    if (!(j == 0 ? want_W : want_E)) continue;
    copy_after_sync(res.comm[j], pin + 96 * (1 + slot++), 96);
    normalise_after_sync(res.comm[j], 1, gens->curve);
  }
}

// 1 = the caller's point is the same group element as the computed one, 0 = it is not
static uint64_t same_point(int curve, const uint8_t* computed96, const void* given96) {
  uint8_t g[96];
  std::memcpy(g, given96, 96);
  vdfgpu_point_normalise_host(curve, g, 1);   // Jacobian of any Z -> (x, y, 1) or (0, 0, 0), as `computed96` is
  return std::memcmp(g, computed96, 96) == 0 ? 1 : 0;
}

// runs after guarded() has waited: fills the report (2 = commitment not checked)
static int sat_report(int rc, const SatResult& res, const vdfgpu_gens* gens, const void* comm_W, const void* comm_E,
                      uint64_t* report4) {
  if (rc != VDFGPU_OK) return rc;
  report4[0] = res.counts[0];
  report4[1] = res.counts[1];
  report4[2] = comm_W ? same_point(gens->curve, res.comm[0], comm_W) : 2;
  report4[3] = comm_E ? same_point(gens->curve, res.comm[1], comm_E) : 2;
  return VDFGPU_OK;
}

}  // namespace vdf

using namespace vdf;

extern "C" {
#pragma GCC visibility push(default)

int vdfgpu_r1cs_create(int field, size_t num_cons, size_t num_vars, size_t num_io,
                       const uint64_t* a_rows, const uint64_t* a_cols, const void* a_vals32, size_t a_nnz,
                       const uint64_t* b_rows, const uint64_t* b_cols, const void* b_vals32, size_t b_nnz,
                       const uint64_t* c_rows, const uint64_t* c_cols, const void* c_vals32, size_t c_nnz,
                       vdfgpu_r1cs** out) {
  return guarded([&] {
    if (!out) throw ArgError("r1cs_create: null out");
    with_field(field, "r1cs_create", [](auto) {});
    if (num_cons == 0 || num_cons >= (1ull << 30) || num_vars >= (1ull << 31)) throw ArgError("r1cs_create: bad dimensions");
    const uint64_t* rows[3] = {a_rows, b_rows, c_rows};
    const uint64_t* cols[3] = {a_cols, b_cols, c_cols};
    const uint8_t* vals[3] = {(const uint8_t*)a_vals32, (const uint8_t*)b_vals32, (const uint8_t*)c_vals32};
    size_t nnzs[3] = {a_nnz, b_nnz, c_nnz};
    size_t nnz = a_nnz + b_nnz + c_nnz;
    if (nnz >= (1ull << 32)) throw ArgError("r1cs_create: too many non-zeros");
    const size_t ncols = num_vars + 1 + num_io;
    HostCsr csr;
    try {
      csr = coo_to_csr(num_cons, ncols, rows, cols, vals, nnzs);
    } catch (const std::invalid_argument& e) {
      throw ArgError(std::string("r1cs_create: ") + e.what());
    }
    require_ready();
    const size_t R = 3 * num_cons;
    std::vector<uint32_t>& row_ptr = csr.row_ptr;
    std::vector<uint32_t>& col = csr.col;
    std::vector<uint8_t>& val = csr.val;
    std::unique_ptr<vdfgpu_r1cs> s(new vdfgpu_r1cs());
    s->field = field;
    s->cons = (uint32_t)num_cons;
    s->vars = (uint32_t)num_vars;
    s->io = (uint32_t)num_io;
    s->nnz = nnz;
    VDF_CUDA_CHECK(cudaMalloc((void**)&s->row_ptr, (R + 1) * 4));
    VDF_CUDA_CHECK(cudaMalloc((void**)&s->col, (nnz ? nnz : 1) * 4));
    VDF_CUDA_CHECK(cudaMalloc((void**)&s->val, (nnz ? nnz : 1) * 32));
    h2d(s->row_ptr, row_ptr.data(), (R + 1) * 4, cur_stream());
    h2d(s->col, col.data(), nnz * 4, cur_stream());
    h2d(s->val, val.data(), nnz * 32, cur_stream());
    const HostCsc csc = csr_to_csc(csr, ncols);
    s->n_heavy = (uint32_t)csc.heavy.size();
    VDF_CUDA_CHECK(cudaMalloc((void**)&s->col_ptr, (ncols + 1) * 4));
    VDF_CUDA_CHECK(cudaMalloc((void**)&s->csc_row, (nnz ? nnz : 1) * 4));
    VDF_CUDA_CHECK(cudaMalloc((void**)&s->csc_val, (nnz ? nnz : 1) * 32));
    VDF_CUDA_CHECK(cudaMalloc((void**)&s->heavy, (s->n_heavy ? s->n_heavy : 1) * 4));
    h2d(s->col_ptr, csc.col_ptr.data(), (ncols + 1) * 4, cur_stream());
    h2d(s->csc_row, csc.srow.data(), nnz * 4, cur_stream());
    h2d(s->csc_val, csc.val.data(), nnz * 32, cur_stream());
    h2d(s->heavy, csc.heavy.data(), (size_t)s->n_heavy * 4, cur_stream());
    sync_after_unlock(cur_stream());
    *out = s.release();
  });
}

int vdfgpu_r1cs_destroy(vdfgpu_r1cs* s) {
  return guarded([&] {
    if (!s) return;
    if (s->refs > 0) throw StateError("r1cs_destroy: a running instance still uses this shape (destroy it first)");
    if (ctx().ready) {
      VDF_CUDA_CHECK(cudaSetDevice(ctx().device));
      cudaDeviceSynchronize();
    }
    delete s;
  });
}

int vdfgpu_multiply_vec(const vdfgpu_r1cs* s, const void* z_host, void* Az_host, void* Bz_host, void* Cz_host) {
  return guarded([&] {
    if (!s || !z_host || !Az_host || !Bz_host || !Cz_host) throw ArgError("multiply_vec: null pointer");
    require_ready();
    CudaLaunch L = api_launch(cur_stream());
    size_t nz = (size_t)s->vars + 1 + s->io;
    DevBuf<fe> z(nz, cur_stream()), out(3 * (size_t)s->cons, cur_stream());
    h2d(z.p, z_host, nz * 32, cur_stream());
    ZView zv{z.p, z.p + s->vars, z.p + s->vars + 1};
    launch_multiply_vec(L, s, zv, out.p, out.p + s->cons, out.p + 2 * (size_t)s->cons);
    d2h(Az_host, out.p, (size_t)s->cons * 32, cur_stream());
    d2h(Bz_host, out.p + s->cons, (size_t)s->cons * 32, cur_stream());
    d2h(Cz_host, out.p + 2 * (size_t)s->cons, (size_t)s->cons * 32, cur_stream());
    sync_after_unlock(cur_stream());
  });
}

int vdfgpu_commit_T(const vdfgpu_r1cs* s, vdfgpu_gens* gens, const void* W1_host, const void* u1_host,
                    const void* X1_host, const void* W2_host, const void* X2_host, void* T_host,
                    void* comm_T_point96_host) {
  return guarded([&] {
    if (!s || !W1_host || !u1_host || !W2_host) throw ArgError("commit_T: null pointer");
    if (s->io && (!X1_host || !X2_host)) throw ArgError("commit_T: null X");
    if (gens && !comm_T_point96_host) throw ArgError("commit_T: null commitment output");
    if (gens) {
      check_gens_field(s, gens);
      if (gens->n < s->cons) throw ArgError("commit_T: fewer generators than constraints");
    }
    require_ready();
    CudaLaunch L = api_launch(cur_stream());
    const size_t nv = s->vars, io = s->io, nc = s->cons;
    DevBuf<fe> W1(nv ? nv : 1, cur_stream()), W2(nv ? nv : 1, cur_stream()), uX1(1 + io, cur_stream()), uX2(1 + io, cur_stream());
    DevBuf<fe> T(nc, cur_stream());
    DevBuf<jac_t> comm(1, cur_stream());
    h2d(W1.p, W1_host, nv * 32, cur_stream());
    h2d(W2.p, W2_host, nv * 32, cur_stream());
    h2d(uX1.p, u1_host, 32, cur_stream());
    h2d(uX1.p + 1, X1_host, io * 32, cur_stream());
    fe one = host_one(s->field);
    h2d(uX2.p, &one, 32, cur_stream());  // u2 = 1 (fresh instance); pageable 32-byte copy is staged by the driver
    h2d(uX2.p + 1, X2_host, io * 32, cur_stream());
    launch_cross_term(L, s, ZView{W1.p, uX1.p, uX1.p + 1}, ZView{W2.p, uX2.p, uX2.p + 1}, T.p);
    const bool hn = gens && host_normalise_wanted(gens);
    if (gens) {
      msm_on_device(gens, 0, T.p, nc, comm.p, true, nullptr, hn);
      d2h(comm_T_point96_host, comm.p, sizeof(jac_t), cur_stream());
    }
    if (T_host) d2h(T_host, T.p, nc * 32, cur_stream());
    sync_after_unlock(cur_stream());
    if (hn) normalise_after_sync(comm_T_point96_host, 1, gens->curve);
  });
}

int vdfgpu_fold(int field, void* W1_host, const void* W2_host, size_t nW, void* E1_host, const void* T_host,
                size_t nE, const void* r32_host) {
  return guarded([&] {
    with_field(field, "fold", [&](auto f) {
      if (!r32_host || (nW && (!W1_host || !W2_host)) || (nE && (!E1_host || !T_host))) throw ArgError("fold: null pointer");
      if (nW + nE == 0) return;
      require_ready();
      CudaLaunch L = api_launch(cur_stream());
      DevBuf<fe> W1(nW ? nW : 1, cur_stream()), W2(nW ? nW : 1, cur_stream()), E1(nE ? nE : 1, cur_stream()), T(nE ? nE : 1, cur_stream()), r(1, cur_stream());
      h2d(W1.p, W1_host, nW * 32, cur_stream());
      h2d(W2.p, W2_host, nW * 32, cur_stream());
      h2d(E1.p, E1_host, nE * 32, cur_stream());
      h2d(T.p, T_host, nE * 32, cur_stream());
      h2d(r.p, r32_host, 32, cur_stream());
      launch_fold<decltype(f)>(L, W1.p, W2.p, nW, E1.p, T.p, nE, r.p);
      d2h(W1_host, W1.p, nW * 32, cur_stream());
      d2h(E1_host, E1.p, nE * 32, cur_stream());
      sync_after_unlock(cur_stream());
    });
  });
}

int vdfgpu_multiply_vec_dev(const vdfgpu_r1cs* s, const void* W_dev, const void* uX_dev, void* AzBzCz_dev) {
  return guarded([&] {
    if (!s || !uX_dev || !AzBzCz_dev || (s->vars && !W_dev)) throw ArgError("multiply_vec_dev: null pointer");
    require_ready();
    CudaLaunch L = api_launch(cur_stream());
    const fe* ux = reinterpret_cast<const fe*>(uX_dev);
    fe* out = reinterpret_cast<fe*>(AzBzCz_dev);
    launch_multiply_vec(L, s, ZView{reinterpret_cast<const fe*>(W_dev), ux, ux + 1}, out, out + s->cons,
                        out + 2 * (size_t)s->cons);
  });
}

int vdfgpu_r1cs_is_sat_relaxed(const vdfgpu_r1cs* s, vdfgpu_gens* gens, const void* W_host, const void* E_host,
                               const void* u_host, const void* X_host, const void* comm_W96_host,
                               const void* comm_E96_host, uint64_t* report4_host) {
  SatResult res;
  const int rc = guarded([&] {
    if (!s || !W_host || !report4_host) throw ArgError("r1cs_is_sat_relaxed: null pointer");
    if (s->io && !X_host) throw ArgError("r1cs_is_sat_relaxed: null X");
    if (!gens && (comm_W96_host || comm_E96_host)) throw ArgError("r1cs_is_sat_relaxed: commitments given without generators");
    if (comm_E96_host && !E_host) throw ArgError("r1cs_is_sat_relaxed: comm_E given without E");
    if (gens) check_sat_gens(s, gens, "r1cs_is_sat_relaxed");
    require_ready();
    cudaStream_t st = cur_stream();
    const size_t nv = s->vars, io = s->io, nc = s->cons;
    DevBuf<fe> W(nv ? nv : 1, st), E(E_host ? nc : 1, st), uX(1 + io, st);
    h2d_scalars(W.p, W_host, nv * 32, st);
    if (E_host) h2d_scalars(E.p, E_host, nc * 32, st);
    const fe one = host_one(s->field);
    h2d(uX.p, u_host ? u_host : &one, 32, st);   // pageable 32-byte copies are staged before cudaMemcpyAsync returns
    h2d(uX.p + 1, X_host, io * 32, st);
    sat_enqueue(s, gens, W.p, E_host ? E.p : nullptr, uX.p, comm_W96_host != nullptr, comm_E96_host != nullptr, res);
  });
  return sat_report(rc, res, gens, comm_W96_host, comm_E96_host, report4_host);
}

int vdfgpu_r1cs_is_sat_relaxed_dev(const vdfgpu_r1cs* s, const void* W_dev, const void* E_dev, const void* uX_dev,
                                   uint64_t* counts2_dev) {
  return guarded([&] {
    if (!s || !uX_dev || !counts2_dev || (s->vars && !W_dev)) throw ArgError("r1cs_is_sat_relaxed_dev: null pointer");
    require_ready();
    CudaLaunch L = api_launch(cur_stream());
    const fe* ux = reinterpret_cast<const fe*>(uX_dev);
    launch_sat(L, s, ZView{reinterpret_cast<const fe*>(W_dev), ux, ux + 1}, reinterpret_cast<const fe*>(E_dev), counts2_dev);
  });
}

static void launch_bind_rows(CudaLaunch& L, const vdfgpu_r1cs* s, const fe* eq, const fe* coef, fe* eq3, fe* out) {
  const size_t ncols = (size_t)s->vars + 1 + s->io;
  const CscView v = s->col_view();
  with_field(s->field, "r1cs", [&](auto f) {
    using F = decltype(f);
    L.run<128>(3 * (size_t)s->cons, ScaleRowsFn<F>{eq, coef, s->cons, eq3});
    L.run<128>(ncols, BindRowsFn<F>{v, eq3, out});
    if (s->n_heavy) L.run<BindHeavyFn<F>::THREADS>((size_t)s->n_heavy * BindHeavyFn<F>::THREADS, BindHeavyFn<F>{v, eq3, out});
  });
}

int vdfgpu_r1cs_bind_rows(const vdfgpu_r1cs* s, const void* eq_rows_host, const void* r_abc_host, void* out_host) {
  return guarded([&] {
    if (!s || !eq_rows_host || !r_abc_host || !out_host) throw ArgError("r1cs_bind_rows: null pointer");
    require_ready();
    CudaLaunch L = api_launch(cur_stream());
    const size_t ncols = (size_t)s->vars + 1 + s->io;
    DevBuf<fe> eq(s->cons, cur_stream()), coef(3, cur_stream()), eq3(3 * (size_t)s->cons, cur_stream()), out(ncols, cur_stream());
    h2d(eq.p, eq_rows_host, (size_t)s->cons * 32, cur_stream());
    h2d(coef.p, r_abc_host, 96, cur_stream());
    launch_bind_rows(L, s, eq.p, coef.p, eq3.p, out.p);
    d2h(out_host, out.p, ncols * 32, cur_stream());
    sync_after_unlock(cur_stream());
  });
}

int vdfgpu_r1cs_bind_rows_dev(const vdfgpu_r1cs* s, const void* eq_rows_dev, const void* r_abc_dev, void* scratch_dev,
                              void* out_dev) {
  return guarded([&] {
    if (!s || !eq_rows_dev || !r_abc_dev || !scratch_dev || !out_dev) throw ArgError("r1cs_bind_rows_dev: null pointer");
    require_ready();
    CudaLaunch L = api_launch(cur_stream());
    launch_bind_rows(L, s, reinterpret_cast<const fe*>(eq_rows_dev), reinterpret_cast<const fe*>(r_abc_dev),
                     reinterpret_cast<fe*>(scratch_dev), reinterpret_cast<fe*>(out_dev));
  });
}

int vdfgpu_cross_term_dev(const vdfgpu_r1cs* s, const void* W1_dev, const void* uX1_dev, const void* W2_dev,
                          const void* uX2_dev, void* T_dev) {
  return guarded([&] {
    if (!s || !uX1_dev || !uX2_dev || !T_dev || (s->vars && (!W1_dev || !W2_dev))) throw ArgError("cross_term_dev: null pointer");
    require_ready();
    CudaLaunch L = api_launch(cur_stream());
    const fe* u1 = reinterpret_cast<const fe*>(uX1_dev);
    const fe* u2 = reinterpret_cast<const fe*>(uX2_dev);
    launch_cross_term(L, s, ZView{reinterpret_cast<const fe*>(W1_dev), u1, u1 + 1},
                      ZView{reinterpret_cast<const fe*>(W2_dev), u2, u2 + 1}, reinterpret_cast<fe*>(T_dev));
  });
}

int vdfgpu_fold_dev(int field, void* W1_dev, const void* W2_dev, size_t nW, void* E1_dev, const void* T_dev,
                    size_t nE, const void* r32_dev) {
  return guarded([&] {
    with_field(field, "fold_dev", [&](auto f) {
      if (!r32_dev || (nW && (!W1_dev || !W2_dev)) || (nE && (!E1_dev || !T_dev))) throw ArgError("fold_dev: null pointer");
      require_ready();
      CudaLaunch L = api_launch(cur_stream());
      launch_fold<decltype(f)>(L, reinterpret_cast<fe*>(W1_dev), reinterpret_cast<const fe*>(W2_dev), nW,
                               reinterpret_cast<fe*>(E1_dev), reinterpret_cast<const fe*>(T_dev), nE,
                               reinterpret_cast<const fe*>(r32_dev));
    });
  });
}

// ---- device-resident running instance -------------------------------------------------------------------
int vdfgpu_running_create(const vdfgpu_r1cs* s, vdfgpu_gens* gens, vdfgpu_running** out) {
  return guarded([&] {
    if (!s || !gens || !out) throw ArgError("running_create: null pointer");
    check_gens_field(s, gens);
    if (gens->n < s->cons || gens->n < s->vars) throw ArgError("running_create: fewer generators than max(cons, vars)");
    require_ready();
    std::unique_ptr<vdfgpu_running> f(new vdfgpu_running());
    f->shape = s;
    f->gens = gens;
    const size_t nv = s->vars ? s->vars : 1, nc = s->cons, io1 = 1 + s->io;
    VDF_CUDA_CHECK(cudaMalloc((void**)&f->W, nv * 32));
    VDF_CUDA_CHECK(cudaMalloc((void**)&f->W2, nv * 32));
    VDF_CUDA_CHECK(cudaMalloc((void**)&f->E, nc * 32));
    VDF_CUDA_CHECK(cudaMalloc((void**)&f->T, nc * 32));
    VDF_CUDA_CHECK(cudaMalloc((void**)&f->uX, io1 * 32));
    VDF_CUDA_CHECK(cudaMalloc((void**)&f->uX2, io1 * 32));
    VDF_CUDA_CHECK(cudaMalloc((void**)&f->r, 32));
    VDF_CUDA_CHECK(cudaMalloc((void**)&f->comm, 2 * sizeof(jac_t)));
    VDF_CUDA_CHECK(cudaHostAlloc((void**)&f->bounce, 2 * sizeof(jac_t) + io1 * sizeof(fe), cudaHostAllocDefault));
    VDF_CUDA_CHECK(cudaEventCreateWithFlags(&f->done, cudaEventDisableTiming));
    s->refs++;
    gens->refs++;
    *out = f.release();
  });
}

int vdfgpu_running_destroy(vdfgpu_running* f) {
  return guarded([&] {
    if (!f) return;
    if (f->refs > 0) throw StateError("running_destroy: a Spartan proof of this instance is in progress");
    if (ctx().ready) {
      VDF_CUDA_CHECK(cudaSetDevice(ctx().device));
      cudaDeviceSynchronize();
    }
    f->shape->refs--;
    f->gens->refs--;
    delete f;
  });
}

int vdfgpu_running_set(vdfgpu_running* f, const void* W_host, const void* E_host, const void* u_host,
                            const void* X_host) {
  return guarded([&] {
    if (!f || !W_host || !E_host || !u_host) throw ArgError("running_set: null pointer");
    if (f->shape->io && !X_host) throw ArgError("running_set: null X");
    require_ready();
    cudaStream_t st = cur_stream();
    running_after(f, st);
    h2d(f->W, W_host, (size_t)f->shape->vars * 32, st);
    h2d(f->E, E_host, (size_t)f->shape->cons * 32, st);
    h2d(f->uX, u_host, 32, st);
    h2d(f->uX + 1, X_host, (size_t)f->shape->io * 32, st);
    running_done(f, st);
    sync_after_unlock(st);
    f->have_running = true;
    f->have_fresh = false;
  });
}

int vdfgpu_running_get(const vdfgpu_running* f, void* W_host, void* E_host, void* u_host, void* X_host) {
  return guarded([&] {
    if (!f) throw ArgError("running_get: null handle");
    if (!f->have_running) throw StateError("running_get: no running instance set");
    require_ready();
    cudaStream_t st = cur_stream();
    running_after(f, st);
    if (W_host) d2h(W_host, f->W, (size_t)f->shape->vars * 32, st);
    if (E_host) d2h(E_host, f->E, (size_t)f->shape->cons * 32, st);
    if (u_host) d2h(u_host, f->uX, 32, st);
    if (X_host) d2h(X_host, f->uX + 1, (size_t)f->shape->io * 32, st);
    running_done(f, st);
    sync_after_unlock(st);
  });
}

// is_sat_relaxed of the resident running instance: W, E, u, X never leave HBM.  Between running_commit and
// running_finish this is still the running (not yet folded) instance: only W2, uX2 and T have changed.
int vdfgpu_running_check(const vdfgpu_running* f, const void* comm_W96_host, const void* comm_E96_host,
                         uint64_t* report4_host) {
  SatResult res;
  const int rc = guarded([&] {
    if (!f || !report4_host) throw ArgError("running_check: null pointer");
    if (!f->have_running) throw StateError("running_check: no running instance set");
    require_ready();
    running_after(f, cur_stream());
    sat_enqueue(f->shape, f->gens, f->W, f->E, f->uX, comm_W96_host != nullptr, comm_E96_host != nullptr, res);
    running_done(f, cur_stream());
  });
  return sat_report(rc, res, f ? f->gens : nullptr, comm_W96_host, comm_E96_host, report4_host);
}

// uX2 = [1 | X2] in one copy from the instance's pinned staging area (the previous step's copy has long completed:
// every commit ends with a wait)
static void upload_ux2(vdfgpu_running* f, const void* X2_host, cudaStream_t st) {
  const vdfgpu_r1cs* s = f->shape;
  fe* stage = reinterpret_cast<fe*>(f->bounce + 2 * sizeof(jac_t));
  stage[0] = host_one(s->field);
  if (s->io) std::memcpy(stage + 1, X2_host, (size_t)s->io * 32);
  h2d(f->uX2, stage, (1 + (size_t)s->io) * 32, st);
}

// the part of running_commit after W2 / X2 are in place: T, then commit(W2) and commit(T) in one batched pass
static void running_commit_enqueue(vdfgpu_running* f, void* comm_W2_point96_host, void* comm_T_point96_host) {
  cudaStream_t st = cur_stream();
  CudaLaunch L = api_launch(st);
  const vdfgpu_r1cs* s = f->shape;
  launch_cross_term(L, s, ZView{f->W, f->uX, f->uX + 1}, ZView{f->W2, f->uX2, f->uX2 + 1}, f->T);
  const fe* vecs[2] = {f->W2, f->T};
  const size_t lens[2] = {s->vars, s->cons};
  const bool hn = host_normalise_wanted(f->gens);
  msm_batch_on_device(f->gens, vecs, lens, 2, f->comm, hn);
  d2h(f->bounce, f->comm, 2 * sizeof(jac_t), st);      // pinned: asynchronous, waited for outside the lock
  running_done(f, st);
  sync_after_unlock(st);
  copy_after_sync(comm_W2_point96_host, f->bounce, sizeof(jac_t));
  copy_after_sync(comm_T_point96_host, f->bounce + sizeof(jac_t), sizeof(jac_t));
  if (hn) {
    normalise_after_sync(comm_W2_point96_host, 1, f->gens->curve);
    normalise_after_sync(comm_T_point96_host, 1, f->gens->curve);
  }
  f->have_fresh = true;
}

int vdfgpu_running_commit(vdfgpu_running* f, const void* W2_host, const void* X2_host, void* comm_W2_point96_host,
                          void* comm_T_point96_host) {
  return guarded([&] {
    if (!f || !W2_host || !comm_W2_point96_host || !comm_T_point96_host) throw ArgError("running_commit: null pointer");
    if (f->shape->io && !X2_host) throw ArgError("running_commit: null X2");
    if (!f->have_running) throw StateError("running_commit: no running instance set");
    require_ready();
    cudaStream_t st = cur_stream();
    const vdfgpu_r1cs* s = f->shape;
    running_after(f, st);
    h2d(f->W2, W2_host, (size_t)s->vars * 32, st);
    upload_ux2(f, X2_host, st);
    running_commit_enqueue(f, comm_W2_point96_host, comm_T_point96_host);
  });
}

// ---- f1: step-circuit witness generation on the device, feeding commit(W) without passing through the host ----
int vdfgpu_witness_bank_create(int field, const void* z_in_state96_host, uint64_t t, size_t n,
                               vdfgpu_witness_bank** out) {
  return guarded([&] {
    if (!out || !z_in_state96_host) throw ArgError("witness_bank_create: null pointer");
    with_field(field, "witness_bank_create", [&](auto f) {
      if (n == 0 || t == 0 || t >= (1ull << 32)) throw ArgError("witness_bank_create: bad dimensions");
      require_ready();
      std::unique_ptr<vdfgpu_witness_bank> b(new vdfgpu_witness_bank());
      b->field = field;
      b->t = t;
      b->n = n;
      const size_t per = 4 * (size_t)t + 1;
      state_t* d_states = nullptr;
      VDF_CUDA_CHECK(cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking));
      VDF_CUDA_CHECK(cudaEventCreateWithFlags(&b->ready, cudaEventDisableTiming));
      VDF_CUDA_CHECK(cudaMalloc((void**)&b->w, n * per * sizeof(fe)));
      VDF_CUDA_CHECK(cudaMallocAsync((void**)&d_states, n * sizeof(state_t), b->stream));
      CudaLaunch L = api_launch(b->stream);
      h2d(d_states, z_in_state96_host, n * sizeof(state_t), b->stream);
      // one thread per step (the rounds of a step are a sequential chain); 32-thread blocks spread few steps
      // over many SMs.  Runs on the bank's own stream: fold steps of the other curve proceed meanwhile.
      L.run<32>(n, MinRootWitnessFn<decltype(f)>{d_states, t, b->w});
      VDF_CUDA_CHECK(cudaFreeAsync(d_states, b->stream));
      VDF_CUDA_CHECK(cudaEventRecord(b->ready, b->stream));
      // the caller's state array may be reused after return: wait for the upload only if it was asynchronous
      // (pinned memory); pageable copies are staged before cudaMemcpyAsync returns
      cudaPointerAttributes at;
      if (cudaPointerGetAttributes(&at, z_in_state96_host) == cudaSuccess && at.type == cudaMemoryTypeHost)
        sync_after_unlock(b->stream);
      else cudaGetLastError();
      *out = b.release();
    });
  });
}

int vdfgpu_witness_bank_destroy(vdfgpu_witness_bank* b) {
  return guarded([&] {
    if (!b) return;
    if (ctx().ready) {
      VDF_CUDA_CHECK(cudaSetDevice(ctx().device));
      cudaDeviceSynchronize();
    }
    delete b;
  });
}

int vdfgpu_witness_bank_read(const vdfgpu_witness_bank* b, size_t first_step, size_t count, void* out_fe32_host) {
  return guarded([&] {
    if (!b || !out_fe32_host) throw ArgError("witness_bank_read: null pointer");
    if (first_step + count > b->n) throw ArgError("witness_bank_read: step range out of bounds");
    require_ready();
    cudaStream_t st = cur_stream();
    const size_t per = 4 * (size_t)b->t + 1;
    VDF_CUDA_CHECK(cudaStreamWaitEvent(st, b->ready, 0));
    d2h(out_fe32_host, b->w + first_step * per, count * per * sizeof(fe), st);
    sync_after_unlock(st);
  });
}

int vdfgpu_running_commit_step(vdfgpu_running* f, const vdfgpu_witness_bank* bank, size_t step, size_t step_offset,
                               const void* W2_host, const void* X2_host, void* comm_W2_point96_host,
                               void* comm_T_point96_host) {
  return guarded([&] {
    if (!f || !bank || !comm_W2_point96_host || !comm_T_point96_host) throw ArgError("running_commit_step: null pointer");
    const vdfgpu_r1cs* s = f->shape;
    const size_t per = 4 * (size_t)bank->t + 1, nv = s->vars;
    if (bank->field != s->field) throw ArgError("running_commit_step: the bank's field differs from the R1CS field");
    if (step >= bank->n) throw ArgError("running_commit_step: step out of range");
    if (step_offset + per > nv) throw ArgError("running_commit_step: step variables do not fit in W");
    if (nv > per && !W2_host) throw ArgError("running_commit_step: null W2");
    if (s->io && !X2_host) throw ArgError("running_commit_step: null X2");
    if (!f->have_running) throw StateError("running_commit_step: no running instance set");
    require_ready();
    cudaStream_t st = cur_stream();
    const uint8_t* w2 = reinterpret_cast<const uint8_t*>(W2_host);
    running_after(f, st);
    // W2 = [ host part | 4t+1 step variables from the bank | host part ]: the step range never crosses PCIe
    h2d(f->W2, w2, step_offset * 32, st);
    h2d(f->W2 + step_offset + per, w2 + (step_offset + per) * 32, (nv - step_offset - per) * 32, st);
    VDF_CUDA_CHECK(cudaStreamWaitEvent(st, bank->ready, 0));
    d2d(f->W2 + step_offset, bank->w + step * per, per * 32, st);
    upload_ux2(f, X2_host, st);
    running_commit_enqueue(f, comm_W2_point96_host, comm_T_point96_host);
  });
}

int vdfgpu_running_finish(vdfgpu_running* f, const void* r32_host) {
  return guarded([&] {
    if (!f || !r32_host) throw ArgError("running_finish: null pointer");
    if (!f->have_fresh) throw StateError("running_finish: fold_commit has not been called for this step");
    require_ready();
    cudaStream_t st = cur_stream();
    CudaLaunch L = api_launch(st);
    const vdfgpu_r1cs* s = f->shape;
    running_after(f, st);
    h2d(f->r, r32_host, 32, st);
    with_field(s->field, "running_finish", [&](auto F) {
      launch_fold<decltype(F)>(L, f->W, f->W2, s->vars, f->E, f->T, s->cons, f->r);
      // u <- u + r*1, X <- X + r*X2: the same kernel over the (1 + io)-element tail
      launch_fold<decltype(F)>(L, f->uX, f->uX2, 1 + (size_t)s->io, nullptr, nullptr, 0, f->r);
    });
    running_done(f, st);
    // No wait: the next call on this instance, on any stream or thread, waits for f->done.  Only a pinned r32_host
    // would still be in flight after return (pageable copies are staged before cudaMemcpyAsync returns).
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, r32_host) == cudaSuccess && at.type == cudaMemoryTypeHost) sync_after_unlock(st);
    else cudaGetLastError();
    f->have_fresh = false;
  });
}

#pragma GCC visibility pop
}  // extern "C"

// ---- Spartan of the running instance: RelaxedR1CSSNARK::prove [R] (notation: sumcheck.cuh) and the sparse evaluation
// of its verifier --------------------------------------------------------------------------------------------------
namespace vdf {

// the caller's round callback behind sumcheck(): it keeps the challenges of the phase (r_x, then r_y) and rejects a
// non-canonical one, which sumcheck() itself would bind
struct SpartanRounds {
  vdfgpu_round_fn fn;
  void* user;
  int field;
  std::vector<fe> r;
  bool non_canonical = false;
};

template <class F>
static bool canonical_all(const fe* v, size_t n) {
  for (size_t i = 0; i < n; i++)
    if (!F::is_canonical(v[i])) return false;
  return true;
}

static int spartan_round(void* p, size_t round, const void* evals, size_t n_evals, void* r_out) {
  SpartanRounds& s = *static_cast<SpartanRounds*>(p);
  if (s.fn(s.user, round, evals, n_evals, r_out) != 0) return 1;
  fe r;
  std::memcpy(&r, r_out, sizeof(fe));
  s.non_canonical = !(s.field == VDFGPU_FP ? canonical_all<Fp>(&r, 1) : canonical_all<Fq>(&r, 1));
  if (s.non_canonical) return 1;
  s.r.push_back(r);
  return 0;
}

// sumcheck() over the running instance's tables with the caller's callback; the challenges land in rounds.r
static int spartan_sumcheck(SpartanRounds& rounds, fe* const* tables, int n_polys, size_t ell, fe* final_evals) {
  rounds.r.clear();
  const void* t[4] = {tables[0], tables[1], n_polys == 4 ? tables[2] : nullptr, n_polys == 4 ? tables[3] : nullptr};
  const int rc = sumcheck(rounds.field, t, n_polys, false, ell, spartan_round, &rounds, final_evals);
  if (rc != VDFGPU_OK && rounds.non_canonical) set_error("running_spartan_prove: the round callback returned a non-canonical challenge");
  else if (rc != VDFGPU_OK) set_error(std::string("running_spartan_prove: ") + vdfgpu_last_error());
  return rc;
}

static const char* const SPARTAN_STAGE[3] = {"OUTER", "EVAL", "IPA"};

// one claims callback, outside the lock: every value it returns must be canonical
static int spartan_claims(int field, vdfgpu_spartan_claims_fn fn, void* user, int stage, const fe* in, size_t n_in,
                          fe* out, size_t n_out) {
  if (fn(user, stage, in, n_in, out, n_out) != 0) {
    set_error(std::string("running_spartan_prove: the claims callback failed at stage ") + SPARTAN_STAGE[stage]);
    return VDFGPU_ERR_STATE;
  }
  if (!(field == VDFGPU_FP ? canonical_all<Fp>(out, n_out) : canonical_all<Fq>(out, n_out))) {
    set_error(std::string("running_spartan_prove: the claims callback returned a non-canonical value at stage ") +
              SPARTAN_STAGE[stage]);
    return VDFGPU_ERR_STATE;
  }
  return VDFGPU_OK;
}

// The call's device buffers, carved from one stream-ordered allocation.  Az..D are contiguous: once the outer claims
// are out they hold the inner tables (Mp over Az, Bz; zp over Cz, D), and eqt then holds eq(r_y').
struct SpartanBufs {
  fe* block = nullptr;
  fe *W, *E, *uX, *Az, *Bz, *Cz, *D, *eqt, *eqx, *r, *eq3, *Mc, *coef, *partial, *res;
  void carve(const vdfgpu_r1cs* s, const PaddedLayout& pad, cudaStream_t st) {
    const size_t m = pad.m, ncols = (size_t)s->vars + 1 + s->io, npart = (size_t)148 * 8 * 3;
    const size_t total = 9 * m + (1 + s->io) + (pad.ell_x + 1) + 3 * (size_t)s->cons + ncols + 3 + npart + 3;
    VDF_CUDA_CHECK(cudaMallocAsync((void**)&block, total * sizeof(fe), st));
    fe* p = block;
    for (fe** q : {&W, &E, &Az, &Bz, &Cz, &D, &eqt, &eqx}) { *q = p; p += m; }
    uX = p; p += 1 + s->io;
    r = p; p += pad.ell_x + 1;
    eq3 = p; p += 3 * (size_t)s->cons;
    Mc = p; p += ncols;
    coef = p; p += 3;
    partial = p; p += npart;
    res = p;
  }
};

// the m-entry zero-padded copy of n elements at src
static void padded_copy(fe* dst, const fe* src, size_t n, size_t m, cudaStream_t st) {
  d2d(dst, src, n * sizeof(fe), st);
  if (m > n) VDF_CUDA_CHECK(cudaMemsetAsync(dst + n, 0, (m - n) * sizeof(fe), st));
}

// K inner products on the device, read back into out_host after the wait
template <class F, int K>
static void spartan_dots(const MultiDot<K>& d, size_t n, const SpartanBufs& b, fe* out_host, cudaStream_t st) {
  multi_dot_enqueue<F, K>(st, d, n, b.partial, b.res);
  fe* pin = pinned_evals();
  d2h(pin, b.res, K * sizeof(fe), st);
  sync_after_unlock(st);
  copy_after_sync(out_host, pin, K * sizeof(fe));
}

// vdfgpu_running_spartan_prove.  Like ipa_prove, a sequence of guarded() sections with the caller's callbacks between
// them; the two sum-checks and the opening are sumcheck() and ipa_prove() themselves.  The shape, the IPA set and the
// instance stay referenced from the first section to the last, so destroying any of them meanwhile is refused.
static int running_spartan_prove(vdfgpu_running* f, vdfgpu_gens* g, const void* tau_host, vdfgpu_round_fn sc_round,
                                 vdfgpu_spartan_claims_fn claims, vdfgpu_ipa_round_fn ipa_round, void* user,
                                 void* a_hat_host) {
  const vdfgpu_r1cs* s = nullptr;
  PaddedLayout pad{};
  SpartanBufs b;
  bool holds = false;
  int rc = guarded([&] {
    if (!f || !g || !tau_host || !sc_round || !claims || !ipa_round || !a_hat_host)
      throw ArgError("running_spartan_prove: null pointer");
    s = f->shape;
    check_gens_field(s, g, "running_spartan_prove: the IPA set: ");
    pad = PaddedLayout::of(s->cons, s->vars, s->io);
    if (!pad.fits()) throw ArgError("running_spartan_prove: 1 + num_io exceeds the padded size m");
    if (g->n < pad.m + 1) throw ArgError("running_spartan_prove: the IPA set needs at least m + 1 points");
    if (!f->have_running) throw StateError("running_spartan_prove: no running instance set");
    require_ready();
    cudaStream_t st = cur_stream();
    CudaLaunch L = api_launch(st);
    b.carve(s, pad, st);
    s->refs++;
    g->refs++;
    f->refs++;
    holds = true;
    // the snapshot: from here on nothing reads the instance, so a later fold step cannot change the proof
    running_after(f, st);
    padded_copy(b.W, f->W, s->vars, pad.m, st);
    padded_copy(b.E, f->E, s->cons, pad.m, st);
    d2d(b.uX, f->uX, (1 + (size_t)s->io) * sizeof(fe), st);
    running_done(f, st);
    h2d(b.r, tau_host, pad.ell_x * sizeof(fe), st);
    with_field(s->field, "running_spartan_prove", [&](auto F) {
      using Fd = decltype(F);
      eq_evals_enqueue<Fd>(L, b.r, pad.ell_x, b.eqt);
      L.run<128>(pad.m, OuterTablesFn<Fd>{s->view(), ZView{b.W, b.uX, b.uX + 1}, b.E, b.Az, b.Bz, b.Cz, b.D});
    });
    // a pinned tau_host may still be in flight: the outer sum-check's first read-back waits for it
  });
  const int field = s ? s->field : 0;
  SpartanRounds rounds{sc_round, user, field, {}, false};
  fe fin[4], dots[2], r_abc[3];   // final evaluations, (claim_Cz, eval_E), (r_A, r_B, r_C)
  std::vector<fe> r_x;
  // outer sum-check -> r_x, claim_Az, claim_Bz; then claim_Cz and eval_E, and the OUTER stage
  if (rc == VDFGPU_OK) {
    fe* t[4] = {b.eqt, b.Az, b.Bz, b.D};
    rc = spartan_sumcheck(rounds, t, 4, pad.ell_x, fin);
    r_x = rounds.r;
  }
  if (rc == VDFGPU_OK)
    rc = guarded([&] {
      require_ready();
      cudaStream_t st = cur_stream();
      CudaLaunch L = api_launch(st);
      h2d(b.r, r_x.data(), pad.ell_x * sizeof(fe), st);   // pageable: staged before cudaMemcpyAsync returns
      with_field(field, "running_spartan_prove", [&](auto F) {
        using Fd = decltype(F);
        eq_evals_enqueue<Fd>(L, b.r, pad.ell_x, b.eqx);
        spartan_dots<Fd, 2>(MultiDot<2>{{b.Cz, b.E}, {b.eqx, b.eqx}, {pad.m, pad.m}}, pad.m, b, dots, st);
      });
    });
  if (rc == VDFGPU_OK) {
    const fe in[4] = {fin[1], fin[2], dots[0], dots[1]};
    rc = spartan_claims(field, claims, user, VDFGPU_SPARTAN_OUTER, in, 4, r_abc, 3);
  }
  // inner tables and inner sum-check -> r_y
  if (rc == VDFGPU_OK)
    rc = guarded([&] {
      require_ready();
      cudaStream_t st = cur_stream();
      CudaLaunch L = api_launch(st);
      h2d(b.coef, r_abc, sizeof(r_abc), st);
      launch_bind_rows(L, s, b.eqx, b.coef, b.eq3, b.Mc);
      with_field(field, "running_spartan_prove", [&](auto F) {
        L.run<256>(2 * pad.m, PaddedScatterFn<decltype(F)>{pad, b.Mc, ZView{b.W, b.uX, b.uX + 1}, b.Az, b.Cz});
      });
    });
  if (rc == VDFGPU_OK) {
    fe* t[2] = {b.Az, b.Cz};
    rc = spartan_sumcheck(rounds, t, 2, pad.ell_x + 1, fin);
  }
  // eval_W, the cross term T, and the EVAL stage
  fe ev[3];   // eval_W, <E, eq(r_y')>, <W, eq(r_x)>
  if (rc == VDFGPU_OK)
    rc = guarded([&] {
      require_ready();
      cudaStream_t st = cur_stream();
      CudaLaunch L = api_launch(st);
      h2d(b.r, rounds.r.data() + 1, pad.ell_x * sizeof(fe), st);   // r_y' = r_y[1..]
      with_field(field, "running_spartan_prove", [&](auto F) {
        using Fd = decltype(F);
        eq_evals_enqueue<Fd>(L, b.r, pad.ell_x, b.eqt);
        spartan_dots<Fd, 3>(MultiDot<3>{{b.W, b.E, b.W}, {b.eqt, b.eqt, b.eqx}, {pad.m, pad.m, pad.m}}, pad.m, b, ev,
                            st);
      });
    });
  fe rho, c, u_scale;
  if (rc == VDFGPU_OK) {
    with_field(field, "running_spartan_prove", [&](auto F) {
      using Fd = decltype(F);
      ev[1] = Fd::add(ev[1], ev[2]);   // T
    });
    rc = spartan_claims(field, claims, user, VDFGPU_SPARTAN_EVAL, ev, 2, &rho, 1);
  }
  // the joint claim: a = E + rho W and b = eq(r_x) + rho eq(r_y') in place of E and eq(r_x), c on the host
  if (rc == VDFGPU_OK)
    rc = guarded([&] {
      require_ready();
      CudaLaunch L = api_launch(cur_stream());
      with_field(field, "running_spartan_prove", [&](auto F) {
        using Fd = decltype(F);
        const fe eval_E = dots[1], T = ev[1], eval_W = ev[0];
        c = Fd::add(eval_E, Fd::mul(rho, Fd::add(T, Fd::mul(rho, eval_W))));
        L.run<256>(pad.m, IpaJoinFn<Fd>{b.E, b.W, b.eqx, b.eqt, rho, b.E, b.eqx});
      });
    });
  if (rc == VDFGPU_OK) rc = spartan_claims(field, claims, user, VDFGPU_SPARTAN_IPA, &c, 1, &u_scale, 1);
  // the opening; ipa_prove validates nothing the checks above have not (its set holds m + 1 points)
  if (rc == VDFGPU_OK) {
    rc = ipa_prove(g, b.E, b.eqx, false, pad.ell_x, &u_scale, ipa_round, user, a_hat_host);
    if (rc != VDFGPU_OK) set_error(std::string("running_spartan_prove: ") + vdfgpu_last_error());
  }
  std::string keep = rc == VDFGPU_OK ? std::string() : std::string(vdfgpu_last_error());
  guarded([&] {
    if (holds) {
      s->refs--;
      g->refs--;
      f->refs--;
    }
    if (b.block && ctx().ready) cudaFreeAsync(b.block, cur_stream());
  });
  if (rc != VDFGPU_OK) set_error(keep);
  return rc;
}

// vdfgpu_r1cs_evaluate: (A, B, C)(r_x, r_y) = sum_x eq(r_x, x) sum_y M[x, y] eq(r_y, y) over the padded layout: the
// rows' products with eq(r_y) read through the padded column map (MultiplyVecFn over PaddedLayout::view), then one
// three-output pass against eq(r_x)
template <class F>
static void r1cs_evaluate_enqueue(const vdfgpu_r1cs* s, const PaddedLayout& pad, const void* rx_host,
                                  const void* ry_host, void* out3_host) {
  cudaStream_t st = cur_stream();
  CudaLaunch L = api_launch(st);
  const size_t nc = s->cons;
  DevBuf<fe> r(2 * (size_t)pad.ell_x + 1, st), eqx(pad.m, st), eqy(2 * pad.m, st), rows(3 * nc, st),
      partial((size_t)148 * 8 * 3, st), res(3, st);
  h2d(r.p, rx_host, pad.ell_x * sizeof(fe), st);
  h2d(r.p + pad.ell_x, ry_host, (pad.ell_x + 1) * sizeof(fe), st);
  eq_evals_enqueue<F>(L, r.p, pad.ell_x, eqx.p);
  eq_evals_enqueue<F>(L, r.p + pad.ell_x, pad.ell_x + 1, eqy.p);
  launch_multiply_vec(L, s, pad.view(eqy.p), rows.p, rows.p + nc, rows.p + 2 * nc);
  multi_dot_enqueue<F, 3>(st, MultiDot<3>{{rows.p, rows.p + nc, rows.p + 2 * nc}, {eqx.p, eqx.p, eqx.p}, {nc, nc, nc}},
                          pad.m, partial.p, res.p);
  fe* pin = pinned_evals();
  d2h(pin, res.p, 3 * sizeof(fe), st);
  sync_after_unlock(st);
  copy_after_sync(out3_host, pin, 3 * sizeof(fe));
}

// ---- the sparse evaluation of k proofs in one pass, and RelaxedR1CSSNARK::verify of k proofs in one call -------------
// pinned landing zone of the batched evaluation's 3k values, one per calling thread (its previous call has been waited
// for), grown on demand
static fe* pinned_abc(size_t count) {
  static thread_local fe* p = nullptr;
  static thread_local size_t cap = 0;
  if (count > cap) {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    VDF_CUDA_CHECK(cudaHostAlloc((void**)&p, count * sizeof(fe), cudaHostAllocDefault));
    cap = count;
  }
  return p;
}

// (A, B, C)(r_x,q, r_y,q) for q < k (r1cs.cuh): the 4k half tables in one launch, SparseEvalBatchFn over every
// (row, proof), the per-block partials summed per output.  rx: [k][ell_x], ry: [k][ell_x + 1] on the host (pageable:
// staged before the copies return); out_host (pinned) receives [k][3] behind the caller's wait.
template <class F>
static void r1cs_evaluate_batch_enqueue(const vdfgpu_r1cs* s, const PaddedLayout& pad, size_t k, const fe* rx,
                                        const fe* ry, fe* out_host, cudaStream_t st) {
  CudaLaunch L = api_launch(st);
  const EqHalves h = EqHalves::of(pad.ell_x);
  uint32_t kq_log = 0;
  while (kq_log < 5 && ((size_t)1 << kq_log) < k) kq_log++;
  const uint32_t gy = (uint32_t)((k + (1u << kq_log) - 1) >> kq_log);
  const size_t rows_per_block = (size_t)SE_BLOCK >> kq_log, need = (s->cons + rows_per_block - 1) / rows_per_block;
  const uint32_t gx = (uint32_t)std::max<size_t>(1, std::min<size_t>(need, std::max<size_t>(1, 148 * 8 / gy)));
  const size_t nx = k * pad.ell_x, ny = k * (pad.ell_x + 1);
  DevBuf<fe> r(nx + ny, st), tables(k * h.per, st), partial((size_t)gx * k * 3, st), res(3 * k, st);
  h2d(r.p, rx, nx * sizeof(fe), st);
  h2d(r.p + nx, ry, ny * sizeof(fe), st);
  L.run<256>(k * h.per, EqHalfTablesBatchFn<F>{r.p, r.p + nx, pad.ell_x, h, tables.p});
  sparse_eval_batch_kernel<F><<<dim3(gx, gy), SE_BLOCK, 0, st>>>(SparseEvalBatchFn<F>{s->view(), pad, h, tables.p, k},
                                                                 kq_log, partial.p);
  sc_column_sum_kernel<F><<<(unsigned)(3 * k), SC_BLOCK, 0, st>>>(partial.p, gx, 3 * k, res.p);
  VDF_CUDA_CHECK(cudaGetLastError());
  ctx().launches += 2;
  d2h(out_host, res.p, 3 * k * sizeof(fe), st);
}

// Offsets in the records of vdfgpu_spartan_verify_batch (include/vdfgpu.h), ell = ell_x
struct SpartanRecords {
  size_t ell;
  size_t proof_fes() const { return 5 * ell + 9; }
  size_t chal_fes() const { return 4 * ell + 6; }
  size_t points() const { return 2 * ell + 2; }
  // proof: outer rounds (e0, e2, e3) x ell, claim_Az, claim_Bz, claim_Cz, eval_E, inner rounds (e0, e2) x (ell + 1),
  // eval_W, T, a_hat
  size_t claims() const { return 3 * ell; }
  size_t inner() const { return 3 * ell + 4; }
  size_t eval_W() const { return 5 * ell + 6; }
  size_t a_hat() const { return 5 * ell + 8; }
  // challenges: tau x ell, r_x x ell, r_A, r_B, r_C, r_y x (ell + 1), rho, u_scale, the IPA's r_j x ell
  size_t r_x() const { return ell; }
  size_t r_abc() const { return 2 * ell; }
  size_t r_y() const { return 2 * ell + 3; }
  size_t rho() const { return 3 * ell + 4; }
  size_t ipa() const { return 3 * ell + 6; }
};

// What the host derives from k proofs: admit[q] = well-formed and every host check passed; the opening's arrays for
// ipa_verify_batch (zero for a proof not admitted); the inner final claim and z(r_y) the device's (A, B, C) completes
struct SpartanVerifyPlan {
  std::vector<uint8_t> admit;
  std::vector<fe> r, a_hat, c, b_hat, u_scale, coef;   // [k][ell], [k] x 4, [k][2] = (rho, 1): comm_W, comm_E
  std::vector<fe> inner_final, z_ry;                   // [k]
};

// The host checks of proof q, O(ell + io) field operations: canonical values, both sum-checks round by round
// (interpolation on 0..3 and 0..2 with the denominators inverted once per call), eq(tau, r_x), the outer final claim,
// eval_X and z(r_y), c and b_hat (r_inv: the IPA challenges' inverses).  The inner final claim waits for (A, B, C).
template <class F>
static void spartan_host_check(const SpartanRecords& R, uint32_t io, const fe* inst, const fe* pf, const fe* ch,
                               const fe* r_inv, const fe (&inv)[2], SpartanVerifyPlan& v, size_t q) {
  const size_t ell = R.ell;
  if (!canonical_all<F>(pf, R.proof_fes()) || !canonical_all<F>(inst, 1 + (size_t)io)) return;
  const fe one = F::one(), two = F::add(one, one), three = F::add(two, one);
  const fe inv2 = inv[0], inv6 = inv[1];
  // claim' = the degree-3 (or 2) interpolant through (0, e0), (1, claim - e0), (2, e2) [, (3, e3)] at r
  auto next = [&](const fe* e, int deg, const fe& claim, const fe& r) {
    const fe y1 = F::sub(claim, e[0]);
    const fe a0 = r, a1 = F::sub(r, one), a2 = F::sub(r, two);
    if (deg == 2)   // y0 a1 a2 / 2 - y1 a0 a2 + y2 a0 a1 / 2
      return F::add(F::sub(F::mul(F::mul(e[0], F::mul(a1, a2)), inv2), F::mul(y1, F::mul(a0, a2))),
                    F::mul(F::mul(e[1], F::mul(a0, a1)), inv2));
    const fe a3 = F::sub(r, three);   // -y0 a1 a2 a3 / 6 + y1 a0 a2 a3 / 2 - y2 a0 a1 a3 / 2 + y3 a0 a1 a2 / 6
    const fe t0 = F::mul(F::mul(e[0], F::mul(a1, F::mul(a2, a3))), inv6);
    const fe t1 = F::mul(F::mul(y1, F::mul(a0, F::mul(a2, a3))), inv2);
    const fe t2 = F::mul(F::mul(e[1], F::mul(a0, F::mul(a1, a3))), inv2);
    const fe t3 = F::mul(F::mul(e[2], F::mul(a0, F::mul(a1, a2))), inv6);
    return F::add(F::sub(F::sub(t1, t0), t2), t3);
  };
  const fe* tau = ch;
  const fe* rx = ch + R.r_x();
  const fe* ry = ch + R.r_y();
  const fe u = inst[0];
  fe claim = F::zero(), eq_tau = one;
  for (size_t j = 0; j < ell; j++) {
    claim = next(pf + 3 * j, 3, claim, rx[j]);
    eq_tau = F::mul(eq_tau, F::add(F::mul(tau[j], rx[j]), F::mul(F::sub(one, tau[j]), F::sub(one, rx[j]))));
  }
  const fe* cl = pf + R.claims();   // claim_Az, claim_Bz, claim_Cz, eval_E
  if (!F::eq(claim, F::mul(eq_tau, F::sub(F::sub(F::mul(cl[0], cl[1]), F::mul(u, cl[2])), cl[3])))) return;
  const fe* rabc = ch + R.r_abc();
  claim = F::add(F::add(F::mul(rabc[0], cl[0]), F::mul(rabc[1], cl[1])), F::mul(rabc[2], cl[2]));
  for (size_t j = 0; j <= ell; j++) claim = next(pf + R.inner() + 2 * j, 2, claim, ry[j]);
  // eval_X = sum_{i <= io} (u, X)[i] eq(r_y', i): eq over the b low variables (2^b > io) times prod (1 - r_y'_j) above
  uint32_t b = 0;
  while (((size_t)1 << b) <= io) b++;
  const fe* ryp = ry + 1;
  fe high = one;
  for (size_t j = 0; j + b < ell; j++) high = F::mul(high, F::sub(one, ryp[j]));
  std::vector<fe> eq_lo(1, high);
  for (size_t j = ell - b; j < ell; j++) {
    std::vector<fe> nxt(2 * eq_lo.size());
    for (size_t i = 0; i < eq_lo.size(); i++) {
      nxt[2 * i + 1] = F::mul(eq_lo[i], ryp[j]);
      nxt[2 * i] = F::sub(eq_lo[i], nxt[2 * i + 1]);
    }
    eq_lo.swap(nxt);
  }
  fe eval_X = F::zero();
  for (size_t i = 0; i <= io; i++) eval_X = F::add(eval_X, F::mul(inst[i], eq_lo[i]));
  const fe eval_W = pf[R.eval_W()], T = pf[R.eval_W() + 1], eval_E = cl[3], rho = ch[R.rho()];
  v.inner_final[q] = claim;
  v.z_ry[q] = F::add(F::mul(F::sub(one, ry[0]), eval_W), F::mul(ry[0], eval_X));
  // the opening: c = eval_E + rho T + rho^2 eval_W, b_hat over the terms (1, r_x) and (rho, r_y')
  v.c[q] = F::add(eval_E, F::mul(rho, F::add(T, F::mul(rho, eval_W))));
  const fe* r = ch + R.ipa();
  fe bx = one, by = one;
  for (size_t j = 0; j < ell; j++) {
    bx = F::mul(bx, F::add(F::mul(F::sub(one, rx[j]), r_inv[j]), F::mul(rx[j], r[j])));
    by = F::mul(by, F::add(F::mul(F::sub(one, ryp[j]), r_inv[j]), F::mul(ryp[j], r[j])));
  }
  v.b_hat[q] = F::add(bx, F::mul(rho, by));
  v.a_hat[q] = pf[R.a_hat()];
  v.u_scale[q] = ch[R.rho() + 1];
  v.coef[2 * q] = rho;
  v.coef[2 * q + 1] = one;
  std::copy(r, r + ell, v.r.begin() + q * ell);
  v.admit[q] = 1;
}

// the batched evaluation for the proofs the opening's batch keeps (ipa_verify_batch's hook)
struct SpartanEvalHook {
  const vdfgpu_r1cs* s;
  PaddedLayout pad;
  const fe* chal;
  SpartanRecords R;
  std::vector<size_t> active;
  std::vector<fe> abc;   // [active][3]
};

static void spartan_eval_hook(void* user, const std::vector<size_t>& active, cudaStream_t st) {
  SpartanEvalHook& h = *static_cast<SpartanEvalHook*>(user);
  const size_t ka = active.size(), lx = h.R.ell, ly = lx + 1;
  h.active = active;
  std::vector<fe> rx(ka * lx + 1), ry(ka * ly);
  for (size_t x = 0; x < ka; x++) {
    const fe* ch = h.chal + active[x] * h.R.chal_fes();
    std::copy(ch + h.R.r_x(), ch + h.R.r_x() + lx, rx.begin() + x * lx);
    std::copy(ch + h.R.r_y(), ch + h.R.r_y() + ly, ry.begin() + x * ly);
  }
  fe* pin = pinned_abc(3 * ka);
  with_field(h.s->field, "spartan_verify_batch", [&](auto F) {
    r1cs_evaluate_batch_enqueue<decltype(F)>(h.s, h.pad, ka, rx.data(), ry.data(), pin, st);
  });
  h.abc.resize(3 * ka);
  copy_after_sync(h.abc.data(), pin, 3 * ka * sizeof(fe));
}

// vdfgpu_spartan_verify_batch: the argument checks and the host checks in one guarded() section, then the opening of
// every admitted proof through ipa_verify_batch, whose first section also enqueues the batched evaluation (one wait
// for both), then the inner final claims on the host.  Shape and set stay referenced from the host checks to the end.
static int spartan_verify_batch(const vdfgpu_r1cs* s, vdfgpu_gens* g, size_t k, const fe* inst, const uint8_t* pts,
                                const fe* proof, const fe* chal, const fe* w, uint8_t* ok) {
  PaddedLayout pad{};
  SpartanRecords R{0};
  SpartanVerifyPlan v;
  bool holds = false;
  int rc = guarded([&] {
    if (!s || !g || !inst || !pts || !proof || !chal || !w || !ok) throw ArgError("spartan_verify_batch: null pointer");
    if (k == 0) throw ArgError("spartan_verify_batch: no proofs");
    std::memset(ok, 0, k);
    check_gens_field(s, g, "spartan_verify_batch: the IPA set: ");
    pad = PaddedLayout::of(s->cons, s->vars, s->io);
    if (!pad.fits()) throw ArgError("spartan_verify_batch: 1 + num_io exceeds the padded size m");
    if (g->n < pad.m + 1) throw ArgError("spartan_verify_batch: the IPA set needs at least m + 1 points");
    R.ell = pad.ell_x;
    with_field(s->field, "spartan_verify_batch", [&](auto F) {
      using Fd = decltype(F);
      for (size_t q = 0; q < k; q++) {
        const fe* ch = chal + q * R.chal_fes();
        if (!canonical_all<Fd>(ch, R.chal_fes()))
          throw ArgError("spartan_verify_batch: a challenge of the caller's transcript is non-canonical");
        for (size_t j = 0; j < R.ell; j++)
          if (!usable_challenge<Fd>(ch[R.ipa() + j])) throw ArgError("spartan_verify_batch: an IPA challenge is 0");
        if (!usable_challenge<Fd>(w[q])) throw ArgError("spartan_verify_batch: a weight is 0 or non-canonical");
      }
      std::vector<fe> r_inv(k * R.ell);
      for (size_t q = 0; q < k; q++)
        std::copy(chal + q * R.chal_fes() + R.ipa(), chal + q * R.chal_fes() + R.ipa() + R.ell, r_inv.begin() + q * R.ell);
      std::vector<fe> inv{Fd::add(Fd::one(), Fd::one()), Fd::zero()};   // 1/2, 1/6
      inv[1] = Fd::add(Fd::add(inv[0], inv[0]), inv[0]);
      inv.insert(inv.end(), r_inv.begin(), r_inv.end());
      batch_invert<Fd>(inv);
      const fe inv26[2] = {inv[0], inv[1]};
      const size_t io1 = 1 + (size_t)s->io;
      v.admit.assign(k, 0);
      for (auto* x : {&v.a_hat, &v.c, &v.b_hat, &v.u_scale, &v.inner_final, &v.z_ry}) x->assign(k, Fd::zero());
      v.r.assign(k * R.ell, Fd::one());
      v.coef.assign(2 * k, Fd::zero());
      for (size_t q = 0; q < k; q++)
        spartan_host_check<Fd>(R, s->io, inst + q * io1, proof + q * R.proof_fes(), chal + q * R.chal_fes(),
                               inv.data() + 2 + q * R.ell, inv26, v, q);
    });
    if (std::find(v.admit.begin(), v.admit.end(), 1) == v.admit.end()) return;
    s->refs++;
    g->refs++;
    holds = true;
  });
  SpartanEvalHook hook{s, pad, chal, R, {}, {}};
  std::vector<uint8_t> opened(k, 0), verdict(k, 0);
  if (rc == VDFGPU_OK && holds) {
    IpaVerifyArgs a{pts, pts + 2 * 96, pts + (2 + R.ell) * 96, v.r.data(), v.a_hat.data(), v.c.data(),
                    v.b_hat.data(), v.u_scale.data(), w, 2, R.points(), R.points(), v.coef.data(), v.admit.data()};
    rc = ipa_verify_batch(g, R.ell, k, a, opened.data(), "spartan_verify_batch", spartan_eval_hook, &hook);
  }
  // the inner final claim: (r_A A + r_B B + r_C C)(r_x, r_y) z(r_y); a proof failing it is dropped after the opening,
  // which is sound: the weighted sum passing says nothing in its favour
  if (rc == VDFGPU_OK && holds)
    with_field(s->field, "spartan_verify_batch", [&](auto F) {
      using Fd = decltype(F);
      for (size_t x = 0; x < hook.active.size(); x++) {
        const size_t q = hook.active[x];
        const fe* rabc = chal + q * R.chal_fes() + R.r_abc();
        const fe* abc = hook.abc.data() + 3 * x;
        const fe m = Fd::add(Fd::add(Fd::mul(rabc[0], abc[0]), Fd::mul(rabc[1], abc[1])), Fd::mul(rabc[2], abc[2]));
        verdict[q] = opened[q] && Fd::eq(v.inner_final[q], Fd::mul(m, v.z_ry[q]));
      }
    });
  if (rc == VDFGPU_OK) std::memcpy(ok, verdict.data(), k);
  if (holds) {
    std::string keep = rc == VDFGPU_OK ? std::string() : std::string(vdfgpu_last_error());
    guarded([&] {
      s->refs--;
      g->refs--;
    });
    if (rc != VDFGPU_OK) set_error(keep);
  }
  return rc;
}

}  // namespace vdf

extern "C" {
#pragma GCC visibility push(default)

int vdfgpu_r1cs_evaluate_batch(const vdfgpu_r1cs* s, size_t k, const void* rx_host, const void* ry_host,
                               void* out3_host) {
  return guarded([&] {
    if (!s || !rx_host || !ry_host || !out3_host) throw ArgError("r1cs_evaluate_batch: null pointer");
    if (k == 0) throw ArgError("r1cs_evaluate_batch: no points");
    const PaddedLayout pad = PaddedLayout::of(s->cons, s->vars, s->io);
    if (!pad.fits()) throw ArgError("r1cs_evaluate_batch: 1 + num_io exceeds the padded size m");
    with_field(s->field, "r1cs_evaluate_batch", [&](auto F) {
      require_ready();
      cudaStream_t st = cur_stream();
      fe* pin = pinned_abc(3 * k);
      r1cs_evaluate_batch_enqueue<decltype(F)>(s, pad, k, reinterpret_cast<const fe*>(rx_host),
                                               reinterpret_cast<const fe*>(ry_host), pin, st);
      sync_after_unlock(st);
      copy_after_sync(out3_host, pin, 3 * k * sizeof(fe));
    });
  });
}

int vdfgpu_spartan_verify_batch(const vdfgpu_r1cs* s, vdfgpu_gens* ipa_gens, size_t k, const void* inst32_host,
                                const void* points96_host, const void* proof32_host, const void* chal32_host,
                                const void* w32_host, uint8_t* ok_out_host) {
  auto fes = [](const void* p) { return reinterpret_cast<const fe*>(p); };
  return spartan_verify_batch(s, ipa_gens, k, fes(inst32_host), reinterpret_cast<const uint8_t*>(points96_host),
                              fes(proof32_host), fes(chal32_host), fes(w32_host), ok_out_host);
}

int vdfgpu_running_spartan_prove(vdfgpu_running* f, vdfgpu_gens* ipa_gens, const void* tau_host,
                                 vdfgpu_round_fn sc_round, vdfgpu_spartan_claims_fn claims,
                                 vdfgpu_ipa_round_fn ipa_round, void* user, void* a_hat32_host) {
  return running_spartan_prove(f, ipa_gens, tau_host, sc_round, claims, ipa_round, user, a_hat32_host);
}

int vdfgpu_r1cs_evaluate(const vdfgpu_r1cs* s, const void* rx_host, const void* ry_host, void* out3_host) {
  return guarded([&] {
    if (!s || !rx_host || !ry_host || !out3_host) throw ArgError("r1cs_evaluate: null pointer");
    const PaddedLayout pad = PaddedLayout::of(s->cons, s->vars, s->io);
    if (!pad.fits()) throw ArgError("r1cs_evaluate: 1 + num_io exceeds the padded size m");
    with_field(s->field, "r1cs_evaluate", [&](auto F) {
      require_ready();
      r1cs_evaluate_enqueue<decltype(F)>(s, pad, rx_host, ry_host, out3_host);
    });
  });
}

#pragma GCC visibility pop
}  // extern "C"
