// C ABI, part 3: sum-check building blocks for CompressedSNARK::prove (SURVEY.md section 8f rank 2; reference
// src/nova/proof.rs:360-368 -> nova-snark 0.8 spartan_with_ipa_pc [R]).  Contract: include/vdfgpu.h.
// The interactive part of a sum-check (absorb the round polynomial into the transcript, squeeze the challenge) is
// host work that belongs to the caller: it is a callback invoked once per round, outside the library's lock.
#include <cstring>
#include <vector>

#include "ctx.cuh"
#include "sumcheck.cuh"

namespace vdf {

void upload_constants_sumcheck() { VDF_CUDA_CHECK(upload_field_constants()); }

template <class F>
static void eq_evals_enqueue(CudaLaunch& L, const fe* r_dev, size_t ell, fe* out_dev) {
  const uint32_t lo_bits = (uint32_t)(ell / 2), hi_bits = (uint32_t)(ell - lo_bits);
  fe* hi = L.alloc<fe>((size_t)1 << hi_bits);
  fe* lo = L.alloc<fe>((size_t)1 << lo_bits);
  L.run<128>((size_t)1 << hi_bits, EqPartFn<F>{r_dev, 0u, hi_bits, hi});
  L.run<128>((size_t)1 << lo_bits, EqPartFn<F>{r_dev, hi_bits, lo_bits, lo});
  L.run<256>((size_t)1 << ell, EqCombineFn<F>{hi, lo, lo_bits, out_dev});
  L.free(hi);
  L.free(lo);
}

struct ScScratch {   // per-call device scratch of the round loop (stream-ordered pool allocations)
  fe* partial = nullptr;   // [grid][3]
  fe* evals = nullptr;     // [4]
};

// Pinned landing zone of the per-round read-backs, one per calling thread: at Nova sizes a round is two small kernels,
// so what a round costs is the round trip to the caller's transcript -- a pageable 96-byte copy is staged by the driver
// (about 10 us), a pinned one is a plain DMA.
static fe* pinned_evals() {
  static thread_local fe* p = nullptr;
  if (!p) VDF_CUDA_CHECK(cudaHostAlloc((void**)&p, 8 * sizeof(fe), cudaHostAllocDefault));
  return p;
}

template <class F>
static void cubic_round_enqueue(cudaStream_t st, const PolySet& P, size_t half, const ScScratch& s) {
  const uint32_t grid = sc_grid(half);
  sc_cubic_round_kernel<F><<<grid, SC_BLOCK, 0, st>>>(P.p[0], P.p[1], P.p[2], P.p[3], half, s.partial);
  sc_final_kernel<F, 3><<<1, SC_BLOCK, 0, st>>>(s.partial, grid, s.evals);
  VDF_CUDA_CHECK(cudaGetLastError());
  ctx().launches += 2;
}

template <class F>
static void quad_round_enqueue(cudaStream_t st, const PolySet& P, size_t half, const ScScratch& s) {
  const uint32_t grid = sc_grid(half);
  sc_quad_round_kernel<F><<<grid, SC_BLOCK, 0, st>>>(P.p[0], P.p[1], half, s.partial);
  sc_final_kernel<F, 2><<<1, SC_BLOCK, 0, st>>>(s.partial, grid, s.evals);
  VDF_CUDA_CHECK(cudaGetLastError());
  ctx().launches += 2;
}

template <class F>
static void dot_enqueue(cudaStream_t st, const fe* a, const fe* b, size_t n, const ScScratch& s) {
  const uint32_t grid = sc_grid(n);
  sc_dot_kernel<F><<<grid, SC_BLOCK, 0, st>>>(a, b, n, s.partial);
  sc_final_kernel<F, 1><<<1, SC_BLOCK, 0, st>>>(s.partial, grid, s.evals);
  VDF_CUDA_CHECK(cudaGetLastError());
  ctx().launches += 2;
}

// Both sum-checks, cubic (4 tables, 3 evaluations) and quadratic (2 tables, 2 evaluations), in both forms: tables on
// the device, bound in place, or on the host (ell <= 30), uploaded first and freed at the end.  Every guarded() section
// ends before the caller's round callback runs, so the tables and the scratch outlive several of them.
static int sumcheck(int field, const void* const* tables, int n_polys, bool on_host, size_t ell, vdfgpu_round_fn fn,
                    void* user, void* final_host) {
  const int n_evals = n_polys == 4 ? 3 : 2;
  PolySet P{{nullptr, nullptr, nullptr, nullptr}};
  ScScratch s;
  int rc = guarded([&] {
    with_field(field, "sumcheck", [](auto) {});
    if (ell > 40 || !final_host || (ell && !fn)) throw ArgError("sumcheck: bad arguments");
    for (int q = 0; q < n_polys; q++)
      if (!tables[q]) throw ArgError("sumcheck: null table");
    if (on_host && ell > 30) throw ArgError("sumcheck: ell too large for the host-table form");
    require_ready();
    cudaStream_t st = cur_stream();
    const size_t bytes = ((size_t)1 << ell) * sizeof(fe);
    for (int q = 0; q < n_polys; q++) {
      if (!on_host) {
        P.p[q] = reinterpret_cast<fe*>(const_cast<void*>(tables[q]));
        continue;
      }
      VDF_CUDA_CHECK(cudaMalloc((void**)&P.p[q], bytes));
      h2d(P.p[q], tables[q], bytes, st);
    }
    VDF_CUDA_CHECK(cudaMallocAsync((void**)&s.partial, (size_t)148 * 8 * 3 * sizeof(fe), st));
    VDF_CUDA_CHECK(cudaMallocAsync((void**)&s.evals, 4 * sizeof(fe), st));
    if (on_host) sync_after_unlock(st);
  });
  size_t len = (size_t)1 << ell;
  for (size_t round = 0; rc == VDFGPU_OK && round < ell; round++) {
    const size_t half = len / 2;
    fe evals[3], r;
    rc = guarded([&] {
      require_ready();
      cudaStream_t st = cur_stream();
      with_field(field, "sumcheck", [&](auto f) {
        if (n_polys == 4) cubic_round_enqueue<decltype(f)>(st, P, half, s);
        else quad_round_enqueue<decltype(f)>(st, P, half, s);
      });
      fe* pin = pinned_evals();
      VDF_CUDA_CHECK(cudaMemcpyAsync(pin, s.evals, n_evals * sizeof(fe), cudaMemcpyDeviceToHost, st));
      VDF_CUDA_CHECK(cudaStreamSynchronize(st));
      for (int k = 0; k < n_evals; k++) evals[k] = pin[k];
    });
    if (rc != VDFGPU_OK) break;
    if (fn(user, round, evals, (size_t)n_evals, &r) != 0) {   // the caller's transcript: outside the lock
      set_error("sumcheck: the round callback failed");
      rc = VDFGPU_ERR_STATE;
      break;
    }
    rc = guarded([&] {
      require_ready();
      CudaLaunch L = api_launch(cur_stream());
      with_field(field, "sumcheck", [&](auto f) {
        L.run<256>((size_t)n_polys * half, BindTopValFn<decltype(f)>{P, half, r});
      });
    });
    len = half;
  }
  if (rc == VDFGPU_OK)
    rc = guarded([&] {
      require_ready();
      cudaStream_t st = cur_stream();
      fe* pin = pinned_evals();
      for (int q = 0; q < n_polys; q++)
        VDF_CUDA_CHECK(cudaMemcpyAsync(pin + q, P.p[q], sizeof(fe), cudaMemcpyDeviceToHost, st));
      VDF_CUDA_CHECK(cudaStreamSynchronize(st));
      std::memcpy(final_host, pin, 32 * (size_t)n_polys);
    });
  std::string keep = rc == VDFGPU_OK ? std::string() : std::string(vdfgpu_last_error());
  guarded([&] {
    if (!ctx().ready) return;
    if (s.partial) cudaFreeAsync(s.partial, cur_stream());
    if (s.evals) cudaFreeAsync(s.evals, cur_stream());
    if (!on_host) return;
    cudaStreamSynchronize(cur_stream());
    for (int q = 0; q < n_polys; q++)
      if (P.p[q]) cudaFree(P.p[q]);
  });
  if (rc != VDFGPU_OK) set_error(keep);
  return rc;
}

// eq(r, x) for every x in {0,1}^ell into out_dev, from the ell challenges at r_host: both forms of vdfgpu_eq_evals
template <class F>
static void eq_evals_from_host(const void* r_host, size_t ell, fe* out_dev, cudaStream_t st) {
  CudaLaunch L = api_launch(st);
  DevBuf<fe> r(ell ? ell : 1, st);
  h2d(r.p, r_host, ell * 32, st);
  eq_evals_enqueue<F>(L, r.p, ell, out_dev);
}

// sum over x of eq(r, x) * poly[x] for a table on the device, into out_host once the wait is over: both forms of
// vdfgpu_poly_evaluate
template <class F>
static void poly_evaluate_enqueue(const fe* poly_dev, const void* r_host, size_t ell, void* out_host, cudaStream_t st) {
  CudaLaunch L = api_launch(st);
  const size_t n = (size_t)1 << ell;
  DevBuf<fe> r(ell ? ell : 1, st), eq(n, st), partial((size_t)148 * 8, st), res(1, st);
  h2d(r.p, r_host, ell * 32, st);
  eq_evals_enqueue<F>(L, r.p, ell, eq.p);
  dot_enqueue<F>(st, eq.p, poly_dev, n, ScScratch{partial.p, res.p});
  d2h(out_host, res.p, sizeof(fe), st);
  sync_after_unlock(st);
}

}  // namespace vdf

using namespace vdf;

extern "C" {
#pragma GCC visibility push(default)

int vdfgpu_eq_evals_dev(int field, const void* r_host, size_t ell, void* out_dev) {
  return guarded([&] {
    with_field(field, "eq_evals", [&](auto f) {
      if (!out_dev || (ell && !r_host) || ell > 40) throw ArgError("eq_evals: bad arguments");
      require_ready();
      eq_evals_from_host<decltype(f)>(r_host, ell, reinterpret_cast<fe*>(out_dev), cur_stream());
      // r_host may be pinned (asynchronous copy still in flight): wait; a pageable copy is already staged
      sync_after_unlock(cur_stream());
    });
  });
}

int vdfgpu_eq_evals(int field, const void* r_host, size_t ell, void* out_host) {
  return guarded([&] {
    with_field(field, "eq_evals", [&](auto f) {
      if (!out_host || (ell && !r_host) || ell > 30) throw ArgError("eq_evals: bad arguments");
      require_ready();
      cudaStream_t st = cur_stream();
      DevBuf<fe> out((size_t)1 << ell, st);
      eq_evals_from_host<decltype(f)>(r_host, ell, out.p, st);
      d2h(out_host, out.p, ((size_t)1 << ell) * sizeof(fe), st);
      sync_after_unlock(st);
    });
  });
}

int vdfgpu_sumcheck_cubic_dev(int field, void* A_dev, void* B_dev, void* C_dev, void* D_dev, size_t ell,
                              vdfgpu_round_fn round_fn, void* user, void* final_evals4_host) {
  const void* t[4] = {A_dev, B_dev, C_dev, D_dev};
  return sumcheck(field, t, 4, false, ell, round_fn, user, final_evals4_host);
}

int vdfgpu_sumcheck_quad_dev(int field, void* A_dev, void* B_dev, size_t ell, vdfgpu_round_fn round_fn, void* user,
                             void* final_evals2_host) {
  const void* t[2] = {A_dev, B_dev};
  return sumcheck(field, t, 2, false, ell, round_fn, user, final_evals2_host);
}

int vdfgpu_sumcheck_cubic(int field, const void* A_host, const void* B_host, const void* C_host, const void* D_host,
                          size_t ell, vdfgpu_round_fn round_fn, void* user, void* final_evals4_host) {
  const void* t[4] = {A_host, B_host, C_host, D_host};
  return sumcheck(field, t, 4, true, ell, round_fn, user, final_evals4_host);
}

int vdfgpu_sumcheck_quad(int field, const void* A_host, const void* B_host, size_t ell, vdfgpu_round_fn round_fn,
                         void* user, void* final_evals2_host) {
  const void* t[2] = {A_host, B_host};
  return sumcheck(field, t, 2, true, ell, round_fn, user, final_evals2_host);
}

int vdfgpu_poly_evaluate_dev(int field, const void* poly_dev, const void* r_host, size_t ell, void* out_host) {
  return guarded([&] {
    with_field(field, "poly_evaluate", [&](auto f) {
      if (!poly_dev || !out_host || (ell && !r_host) || ell > 40) throw ArgError("poly_evaluate: bad arguments");
      require_ready();
      poly_evaluate_enqueue<decltype(f)>(reinterpret_cast<const fe*>(poly_dev), r_host, ell, out_host, cur_stream());
    });
  });
}

int vdfgpu_poly_evaluate(int field, const void* poly_host, const void* r_host, size_t ell, void* out_host) {
  return guarded([&] {
    with_field(field, "poly_evaluate", [&](auto f) {
      if (!poly_host || !out_host || (ell && !r_host) || ell > 30) throw ArgError("poly_evaluate: bad arguments");
      require_ready();
      cudaStream_t st = cur_stream();
      const size_t bytes = ((size_t)1 << ell) * sizeof(fe);
      DevBuf<fe> poly((size_t)1 << ell, st);
      h2d(poly.p, poly_host, bytes, st);
      poly_evaluate_enqueue<decltype(f)>(poly.p, r_host, ell, out_host, st);
    });
  });
}

// ---- inner-product-argument building blocks ------------------------------------------------------------------
int vdfgpu_vec_lincomb(int field, const void* a_host, const void* b_host, size_t n, const void* x32_host,
                       const void* y32_host, void* out_host) {
  return guarded([&] {
    with_field(field, "vec_lincomb", [&](auto f) {
      if (!x32_host || !y32_host || (n && (!a_host || !b_host || !out_host))) throw ArgError("vec_lincomb: null pointer");
      if (!n) return;
      require_ready();
      cudaStream_t st = cur_stream();
      CudaLaunch L = api_launch(st);
      DevBuf<fe> a(n, st), b(n, st), o(n, st), xy(2, st);
      h2d(a.p, a_host, n * 32, st);
      h2d(b.p, b_host, n * 32, st);
      h2d(xy.p, x32_host, 32, st);
      h2d(xy.p + 1, y32_host, 32, st);
      L.run<256>(n, VecLinCombFn<decltype(f)>{a.p, b.p, xy.p, o.p});
      d2h(out_host, o.p, n * 32, st);
      sync_after_unlock(st);
    });
  });
}

int vdfgpu_inner_product(int field, const void* a_host, const void* b_host, size_t n, void* out32_host) {
  return guarded([&] {
    with_field(field, "inner_product", [&](auto f) {
      if (!out32_host || (n && (!a_host || !b_host))) throw ArgError("inner_product: null pointer");
      require_ready();
      cudaStream_t st = cur_stream();
      DevBuf<fe> a(n ? n : 1, st), b(n ? n : 1, st), partial((size_t)148 * 8, st), res(1, st);
      h2d(a.p, a_host, n * 32, st);
      h2d(b.p, b_host, n * 32, st);
      dot_enqueue<decltype(f)>(st, a.p, b.p, n, ScScratch{partial.p, res.p});
      d2h(out32_host, res.p, sizeof(fe), st);
      sync_after_unlock(st);
    });
  });
}

int vdfgpu_points_lincomb(int curve, const void* P_affine72_host, const void* Q_affine72_host, size_t n,
                          const void* w1_32_host, const void* w2_32_host, void* out_affine72_host) {
  return guarded([&] {
    with_curve(curve, "points_lincomb", [&](auto C, auto BF, auto SF) {
      if (!w1_32_host || !w2_32_host || (n && (!P_affine72_host || !Q_affine72_host || !out_affine72_host)))
        throw ArgError("points_lincomb: null pointer");
      if (!n) return;
      require_ready();
      cudaStream_t st = cur_stream();
      CudaLaunch L = api_launch(st);
      DevBuf<uint8_t> raw(2 * n * 72, st);
      DevBuf<affine_t> pq(2 * n, st), out(n, st);
      DevBuf<fe> w(2, st);
      h2d(raw.p, P_affine72_host, n * 72, st);
      h2d(raw.p + n * 72, Q_affine72_host, n * 72, st);
      h2d(w.p, w1_32_host, 32, st);
      h2d(w.p + 1, w2_32_host, 32, st);
      L.run<256>(2 * n, RepackFn{raw.p, pq.p});
      L.run<64>((n + 3) / 4, PointLinCombFn<decltype(C), decltype(BF), decltype(SF)>{pq.p, pq.p + n, w.p, out.p, n});
      L.run<256>(n, UnpackFn{out.p, raw.p});
      d2h(out_affine72_host, raw.p, n * 72, st);
      sync_after_unlock(st);
    });
  });
}

#pragma GCC visibility pop
}  // extern "C"
