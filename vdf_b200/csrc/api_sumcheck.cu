// C ABI, part 3: sum-check building blocks for CompressedSNARK::prove (SURVEY.md section 8f rank 2; reference
// src/nova/proof.rs:360-368 -> nova-snark 0.8 spartan_with_ipa_pc [R]).  Contract: include/vdfgpu.h.
// The interactive part of a sum-check (absorb the round polynomial into the transcript, squeeze the challenge) is
// host work that belongs to the caller: it is a callback invoked once per round, outside the library's lock.
#include <algorithm>
#include <cstring>
#include <vector>

#include "ctx.cuh"
#include "sumcheck.cuh"

namespace vdf {

void upload_constants_sumcheck() { VDF_CUDA_CHECK(upload_field_constants()); }

template <class F>
void eq_evals_enqueue(CudaLaunch& L, const fe* r_dev, size_t ell, fe* out_dev) {
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
// (about 10 us), a pinned one is a plain DMA.  24 elements: the eight points a chunk of vdfgpu_ipa_verify_batch's
// single-proof checks reads back.
fe* pinned_evals() {
  static thread_local fe* p = nullptr;
  if (!p) VDF_CUDA_CHECK(cudaHostAlloc((void**)&p, 24 * sizeof(fe), cudaHostAllocDefault));
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

template <class F, int K>
void multi_dot_enqueue(cudaStream_t st, const MultiDot<K>& d, size_t n, fe* partial, fe* out) {
  const uint32_t grid = sc_grid(n);
  sc_multi_dot_kernel<F, K><<<grid, SC_BLOCK, 0, st>>>(d, n, partial);
  sc_final_kernel<F, K><<<1, SC_BLOCK, 0, st>>>(partial, grid, out);
  VDF_CUDA_CHECK(cudaGetLastError());
  ctx().launches += 2;
}

// the instances other translation units use (ctx.cuh)
template void eq_evals_enqueue<Fp>(CudaLaunch&, const fe*, size_t, fe*);
template void eq_evals_enqueue<Fq>(CudaLaunch&, const fe*, size_t, fe*);
template void multi_dot_enqueue<Fp, 2>(cudaStream_t, const MultiDot<2>&, size_t, fe*, fe*);
template void multi_dot_enqueue<Fq, 2>(cudaStream_t, const MultiDot<2>&, size_t, fe*, fe*);
template void multi_dot_enqueue<Fp, 3>(cudaStream_t, const MultiDot<3>&, size_t, fe*, fe*);
template void multi_dot_enqueue<Fq, 3>(cudaStream_t, const MultiDot<3>&, size_t, fe*, fe*);

// Both sum-checks, cubic (4 tables, 3 evaluations) and quadratic (2 tables, 2 evaluations), in both forms: tables on
// the device, bound in place, or on the host (ell <= 30), uploaded first and freed at the end.  Every guarded() section
// ends before the caller's round callback runs, so the tables and the scratch outlive several of them.
int sumcheck(int field, const void* const* tables, int n_polys, bool on_host, size_t ell, vdfgpu_round_fn fn,
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

// ---- the inner-product argument (notation: sumcheck.cuh) -------------------------------------------------------
struct IpaScratch {   // per-call device scratch of the IPA round loop (stream-ordered pool allocations)
  fe* a = nullptr;         // host form only: the uploaded a and b
  fe* b = nullptr;
  fe* coef[2] = {nullptr, nullptr};   // coef_j and coef_{j+1}, n entries each
  fe* S[2] = {nullptr, nullptr};      // SL, SR: n + 1 entries each, the same pointers every round (graph replay)
  fe* partial = nullptr;   // [grid][2]
  fe* c = nullptr;         // [2] = (c_L, c_R)
  jac_t* out = nullptr;    // [2] = (L, R), un-normalised
  std::vector<void*> all() const { return {a, b, coef[0], coef[1], S[0], S[1], partial, c, out}; }
};

template <class T>
static T* pool_alloc(size_t count, cudaStream_t st) {
  void* p = nullptr;
  VDF_CUDA_CHECK(cudaMallocAsync(&p, count * sizeof(T) + 16, st));
  return reinterpret_cast<T*>(p);
}

// s = coef_0 = [1] into coef[0]
template <class F>
static void ipa_coef_init(fe* coef, cudaStream_t st) {
  const fe one = F::one();
  h2d(coef, &one, sizeof(fe), st);   // pageable source: staged before cudaMemcpyAsync returns
}

// Both forms of vdfgpu_ipa_prove.  Like sumcheck(): every guarded() section ends before the caller's round callback
// runs; a round is (c_L, c_R), the expansion into SL / SR, ONE batched MSM with k = 2 and one 192-byte read-back into
// pinned memory, normalised on the host after the wait (the transcript absorbs canonical points, whatever the set's
// flags); the fold takes r and r^-1 by value.  The call holds a reference on g from its first guarded() section to its
// last, so vdfgpu_gens_destroy from another thread between rounds is refused instead of freeing the points.
int ipa_prove(vdfgpu_gens* g, void* a_in, void* b_in, bool on_host, size_t ell, const void* u_scale_host,
              vdfgpu_ipa_round_fn fn, void* user, void* a_hat_host) {
  IpaScratch s;
  fe u_scale;
  fe* a = reinterpret_cast<fe*>(a_in);
  fe* b = reinterpret_cast<fe*>(b_in);
  const size_t n = ell <= 40 ? (size_t)1 << ell : 0;
  bool holds_g = false;
  int rc = guarded([&] {
    if (!g || !a_in || !b_in || !u_scale_host || !a_hat_host || (ell && !fn)) throw ArgError("ipa_prove: null pointer");
    if (on_host && ell > 30) throw ArgError("ipa_prove: ell too large for the host-vector form");
    if (ell > 40 || g->n < n + 1) throw ArgError("ipa_prove: the generator set needs at least 2^ell + 1 points");
    std::memcpy(&u_scale, u_scale_host, sizeof(fe));
    require_ready();
    g->refs++;
    holds_g = true;
    cudaStream_t st = cur_stream();
    if (on_host) {
      a = s.a = pool_alloc<fe>(n, st);
      b = s.b = pool_alloc<fe>(n, st);
      h2d_scalars(a, a_in, n * sizeof(fe), st);
      h2d_scalars(b, b_in, n * sizeof(fe), st);
    }
    for (int q = 0; q < 2; q++) {
      s.coef[q] = pool_alloc<fe>(n, st);
      s.S[q] = pool_alloc<fe>(n + 1, st);
    }
    s.partial = pool_alloc<fe>((size_t)sc_grid(n / 2) * 2, st);
    s.c = pool_alloc<fe>(2, st);
    s.out = pool_alloc<jac_t>(2, st);
    with_curve(g->curve, "ipa_prove", [&](auto, auto, auto SF) { ipa_coef_init<decltype(SF)>(s.coef[0], st); });
  });
  int cur = 0;
  for (size_t round = 0; rc == VDFGPU_OK && round < ell; round++) {
    const size_t h = (n >> round) / 2, nc = (size_t)1 << round;
    uint8_t LR[2][96];
    fe r, r_inv;
    rc = guarded([&] {
      require_ready();
      cudaStream_t st = cur_stream();
      with_curve(g->curve, "ipa_prove", [&](auto, auto, auto SF) {
        using F = decltype(SF);
        const uint32_t grid = sc_grid(h);
        sc_cross_dot_kernel<F><<<grid, SC_BLOCK, 0, st>>>(a, b, h, s.partial);
        sc_final_kernel<F, 2><<<1, SC_BLOCK, 0, st>>>(s.partial, grid, s.c);
        VDF_CUDA_CHECK(cudaGetLastError());
        ctx().launches += 2;
        CudaLaunch L = api_launch(st);
        L.run<256>(n + 1, IpaExpandFn<F>{a, s.coef[cur], s.c, u_scale, (uint32_t)(ell - round), n, s.S[0], s.S[1]});
      });
      const fe* vecs[2] = {s.S[0], s.S[1]};
      const size_t lens[2] = {n + 1, n + 1};
      msm_batch_on_device(g, vecs, lens, 2, s.out, true);
      fe* pin = pinned_evals();
      d2h(pin, s.out, 2 * sizeof(jac_t), st);
      sync_after_unlock(st);
      copy_after_sync(LR, pin, sizeof(LR));
      normalise_after_sync(LR, 2, g->curve);
    });
    if (rc != VDFGPU_OK) break;
    if (fn(user, round, LR[0], LR[1], &r) != 0) {   // the caller's transcript: outside the lock
      set_error("ipa_prove: the round callback failed");
      rc = VDFGPU_ERR_STATE;
      break;
    }
    if (!with_curve(g->curve, "ipa_prove", [&](auto, auto, auto SF) { return usable_challenge<decltype(SF)>(r); })) {
      set_error("ipa_prove: the round callback returned 0 or a non-canonical challenge");
      rc = VDFGPU_ERR_STATE;
      break;
    }
    rc = guarded([&] {
      require_ready();
      CudaLaunch L = api_launch(cur_stream());
      with_curve(g->curve, "ipa_prove", [&](auto, auto, auto SF) {
        using F = decltype(SF);
        r_inv = F::inv(r);
        L.run<256>(h > nc ? h : nc, IpaFoldFn<F>{a, b, h, s.coef[cur], s.coef[cur ^ 1], nc, r, r_inv});
      });
    });
    cur ^= 1;
  }
  if (rc == VDFGPU_OK)
    rc = guarded([&] {
      require_ready();
      cudaStream_t st = cur_stream();
      fe* pin = pinned_evals();
      d2h(pin, a, sizeof(fe), st);
      sync_after_unlock(st);
      copy_after_sync(a_hat_host, pin, sizeof(fe));
    });
  std::string keep = rc == VDFGPU_OK ? std::string() : std::string(vdfgpu_last_error());
  guarded([&] {
    if (holds_g) g->refs--;
    if (!ctx().ready) return;
    for (void* p : s.all())
      if (p) cudaFreeAsync(p, cur_stream());
  });
  if (rc != VDFGPU_OK) set_error(keep);
  return rc;
}

// G_hat = <s, G[0, 2^ell)>: the s table by ell doubling launches of IpaFoldFn, then one MSM, normalised on the host
template <class F>
static void ipa_gens_hat_enqueue(vdfgpu_gens* g, const fe* r, const fe* r_inv, size_t ell, void* out_host) {
  cudaStream_t st = cur_stream();
  CudaLaunch L = api_launch(st);
  const size_t n = (size_t)1 << ell;
  DevBuf<fe> t0(n, st), t1(n, st);
  DevBuf<jac_t> out(1, st);
  fe* coef[2] = {t0.p, t1.p};
  ipa_coef_init<F>(coef[0], st);
  for (size_t j = 0; j < ell; j++)
    L.run<256>((size_t)1 << j, IpaFoldFn<F>{nullptr, nullptr, 0, coef[j & 1], coef[(j & 1) ^ 1], (size_t)1 << j, r[j],
                                              r_inv[j]});
  msm_on_device(g, 0, coef[ell & 1], n, out.p, true, st, true);
  fe* pin = pinned_evals();
  d2h(pin, out.p, sizeof(jac_t), st);
  sync_after_unlock(st);
  copy_after_sync(out_host, pin, sizeof(jac_t));
  normalise_after_sync(out_host, 1, g->curve);
}

// ---- batch verification of inner-product arguments (notation: sumcheck.cuh) ---------------------------------------
// What the host derives from the well-formed proofs ("active", in order, ka of them; per = terms + 2 ell points each)
struct IpaVerifyPlan {
  size_t per = 0;
  std::vector<size_t> active;
  std::vector<fe> rr;             // r [ka][ell], then r^-1 [ka][ell], then w a_hat [ka]: the IpaHalfTablesFn inputs
  std::vector<fe> last;           // [ka] w u_scale (a_hat b_hat - c): S[n] of proof q alone; the batch's is their sum
  std::vector<uint8_t> pts72;     // [ka][per] the commitment's terms, L_0 .. L_{ell-1}, R_0 .. R_{ell-1} as 72-byte
                                  // affine records
  std::vector<fe> small;          // [ka][per] their scalars -w coef_t, -w r_j^2, -w r_j^-2
};

struct IpaVerifyScratch {   // device buffers of one call, kept for the single-proof checks of a failing batch
  fe* rr = nullptr;
  fe* tables = nullptr;     // all Hi tables, then all Lo tables
  fe* S = nullptr;          // n + 1: the batch
  fe* small = nullptr;      // ka per: the batch
  uint8_t* raw = nullptr;   // the 72-byte records, repacked into pts
  affine_t* pts = nullptr;
  jac_t* out = nullptr;     // [2 MSM_MAX_BATCH + 1]
  fe* S4 = nullptr;         // MSM_MAX_BATCH (n + 1), MSM_MAX_BATCH ka per: the single-proof checks, allocated only
  fe* small4 = nullptr;     // when the batch fails
  std::vector<void*> all() const { return {rr, tables, S, small, raw, pts, out, S4, small4}; }
};

// The host half of the call: the well-formed admitted proofs (the others keep verdict 0), their points checked on the
// curve and written as affine records (one batched inversion for every Z other than 0 and 1; L and R from
// vdfgpu_ipa_prove have Z = 1), r^-1 by one batched inversion, and the scalars of both MSMs.  Challenges and weights
// were checked by the caller.
template <class BF, class SF>
static IpaVerifyPlan ipa_verify_prepare(size_t ell, size_t k, const IpaVerifyArgs& a) {
  std::vector<uint8_t> good(k);   // well-formed so far
  const size_t nt = a.terms, per = nt + 2 * ell;
  const fe one = BF::one(), b = BF::add(BF::add(BF::add(one, one), BF::add(one, one)), one);   // y^2 = x^3 + 5
  auto point = [&](size_t q, size_t i) -> const uint8_t* {
    return i < nt ? a.comm + 96 * (q * a.comm_stride + i)
                  : i < nt + ell ? a.L + 96 * (q * a.lr_stride + i - nt) : a.R + 96 * (q * a.lr_stride + i - nt - ell);
  };
  std::vector<jac_t> P(k * per);   // proof q's points at [q per, (q + 1) per); those not read stay the identity
  for (size_t q = 0; q < k; q++) {
    good[q] = (!a.admit || a.admit[q]) && SF::is_canonical(a.a_hat[q]) && SF::is_canonical(a.c[q]) &&
              SF::is_canonical(a.b_hat[q]) && SF::is_canonical(a.u_scale[q]);
    for (size_t i = 0; good[q] && i < per; i++) {
      jac_t& pt = P[q * per + i];
      std::memcpy(&pt, point(q, i), sizeof(jac_t));
      good[q] = BF::is_canonical(pt.X) && BF::is_canonical(pt.Y) && BF::is_canonical(pt.Z);
      if (!good[q]) pt = jac_t{};   // a non-canonical Z (m itself is one) must not join the shared inversion
    }
  }
  normalise_host<BF>(P.data(), P.size());
  IpaVerifyPlan p;
  p.per = per;
  for (size_t q = 0; q < k; q++) {
    for (size_t i = 0; good[q] && i < per; i++) {
      const jac_t& pt = P[q * per + i];
      if (!BF::is_zero(pt.Z))
        good[q] = BF::eq(BF::mul(pt.Y, pt.Y), BF::add(BF::mul(BF::mul(pt.X, pt.X), pt.X), b));
    }
    if (good[q]) p.active.push_back(q);
  }
  const size_t ka = p.active.size();
  p.rr.resize(ka * (2 * ell + 1));
  p.last.resize(ka);
  p.pts72.assign(ka * per * 72, 0);
  p.small.resize(ka * per);
  fe* r = p.rr.data();
  fe* r_inv = r + ka * ell;
  fe* scale = r_inv + ka * ell;
  for (size_t x = 0; x < ka && ell; x++) std::memcpy(r + x * ell, a.r + p.active[x] * ell, ell * sizeof(fe));
  std::vector<fe> inv(r, r + ka * ell);
  batch_invert<SF>(inv);
  std::copy(inv.begin(), inv.end(), r_inv);
  for (size_t x = 0; x < ka; x++) {
    const size_t q = p.active[x];
    const fe w = a.w[q], nw = SF::neg(w);
    scale[x] = SF::mul(w, a.a_hat[q]);
    p.last[x] = SF::mul(SF::mul(w, a.u_scale[q]), SF::sub(SF::mul(a.a_hat[q], a.b_hat[q]), a.c[q]));
    fe* sm = p.small.data() + x * per;
    for (size_t t = 0; t < nt; t++) sm[t] = a.coef ? SF::mul(nw, a.coef[q * nt + t]) : nw;
    for (size_t j = 0; j < ell; j++) {
      sm[nt + j] = SF::mul(nw, SF::mul(r[x * ell + j], r[x * ell + j]));
      sm[nt + ell + j] = SF::mul(nw, SF::mul(r_inv[x * ell + j], r_inv[x * ell + j]));
    }
    for (size_t i = 0; i < per; i++) {
      const jac_t& pt = P[q * per + i];
      uint8_t* rec = p.pts72.data() + (x * per + i) * 72;
      if (BF::is_zero(pt.Z)) {
        rec[64] = 1;   // the infinity flag
      } else {
        std::memcpy(rec, &pt.X, 32);
        std::memcpy(rec + 32, &pt.Y, 32);
      }
    }
  }
  return p;
}

// the proofs' own points as a transient plain-layout set (the layout vdfgpu_gens_create makes without flags)
static vdfgpu_gens ipa_small_set(int curve, affine_t* pts, size_t count) {
  vdfgpu_gens gs;
  gs.curve = curve;
  gs.n = count;
  gs.W = 1;
  gs.pts = pts;
  return gs;
}

// The weighted sum of all active proofs: Hi / Lo tables, S, the MSM over g, the proofs' points uploaded and
// repacked, the MSM over them, the sum of the two results; one 96-byte read-back into sum_host (normalised on the
// device: the identity is 96 zero bytes)
template <class C, class SF>
static void ipa_verify_batch_enqueue(vdfgpu_gens* g, size_t ell, const IpaVerifyPlan& p, IpaVerifyScratch& s,
                                     void* sum_host) {
  cudaStream_t st = cur_stream();
  CudaLaunch L = api_launch(st);
  const size_t ka = p.active.size(), n = (size_t)1 << ell, ns = p.small.size();
  const uint32_t lo_bits = (uint32_t)(ell / 2), hi_bits = (uint32_t)ell - lo_bits;
  const size_t hi_len = ka << hi_bits, lo_len = ka << lo_bits;
  s.rr = pool_alloc<fe>(p.rr.size(), st);
  s.tables = pool_alloc<fe>(hi_len + lo_len, st);
  s.S = pool_alloc<fe>(n + 1, st);
  s.small = pool_alloc<fe>(ns, st);
  s.raw = pool_alloc<uint8_t>(p.pts72.size(), st);
  s.pts = pool_alloc<affine_t>(ns, st);
  s.out = pool_alloc<jac_t>(2 * MSM_MAX_BATCH + 1, st);
  h2d(s.rr, p.rr.data(), p.rr.size() * sizeof(fe), st);   // pageable sources: staged before cudaMemcpyAsync returns
  h2d(s.small, p.small.data(), ns * sizeof(fe), st);
  h2d(s.raw, p.pts72.data(), p.pts72.size(), st);
  fe last = SF::zero();
  for (const fe& x : p.last) last = SF::add(last, x);
  L.run<256>(hi_len + lo_len, IpaHalfTablesFn<SF>{s.rr, s.rr + ka * ell, s.rr + 2 * ka * ell, (uint32_t)ell, lo_bits,
                                                  ka, s.tables, s.tables + hi_len});
  L.run<256>(n + 1, IpaBatchScalarsFn<SF>{s.tables, s.tables + hi_len, hi_bits, lo_bits, ka, last, s.S});
  msm_on_device(g, 0, s.S, n + 1, s.out, true, st, true);
  L.run<256>(ns, RepackFn{s.raw, s.pts});
  vdfgpu_gens gs = ipa_small_set(g->curve, s.pts, ns);
  msm_on_device(&gs, 0, s.small, ns, s.out + 1, true, st, true, false);
  L.run<32>(32, JacSumFn<C>{s.out, 2, s.out + 2});
  fe* pin = pinned_evals();
  d2h(pin, s.out + 2, sizeof(jac_t), st);
  sync_after_unlock(st);
  copy_after_sync(sum_host, pin, sizeof(jac_t));
}

// Active proofs [first, first + kc), kc <= MSM_MAX_BATCH, each alone: proof q's share of the batch (its S from its
// own Hi / Lo tables, its slice of the small scalars) as kc vectors of one batched MSM over g and one over the small
// set.  out_host receives the kc results over g, then at 4 * 96 bytes the kc over the small set, normalised.
template <class SF>
static void ipa_verify_chunk_enqueue(vdfgpu_gens* g, size_t ell, const IpaVerifyPlan& p, IpaVerifyScratch& s,
                                     size_t first, uint32_t kc, void* out_host) {
  cudaStream_t st = cur_stream();
  CudaLaunch L = api_launch(st);
  const size_t ka = p.active.size(), n = (size_t)1 << ell, ns = p.small.size(), per = p.per;
  const uint32_t lo_bits = (uint32_t)(ell / 2), hi_bits = (uint32_t)ell - lo_bits;
  if (!s.S4) {
    s.S4 = pool_alloc<fe>(MSM_MAX_BATCH * (n + 1), st);
    s.small4 = pool_alloc<fe>(MSM_MAX_BATCH * ns, st);
  }
  std::vector<fe> sm((size_t)kc * ns, SF::zero());
  const fe* vg[MSM_MAX_BATCH];
  const fe* vs[MSM_MAX_BATCH];
  size_t lg[MSM_MAX_BATCH], ls[MSM_MAX_BATCH];
  for (uint32_t j = 0; j < kc; j++) {
    const size_t x = first + j;
    fe* S = s.S4 + j * (n + 1);
    L.run<256>(n + 1, IpaBatchScalarsFn<SF>{s.tables + (x << hi_bits), s.tables + (ka << hi_bits) + (x << lo_bits),
                                            hi_bits, lo_bits, 1, p.last[x], S});
    std::copy(p.small.begin() + x * per, p.small.begin() + (x + 1) * per, sm.begin() + j * ns + x * per);
    vg[j] = S;
    lg[j] = n + 1;
    vs[j] = s.small4 + j * ns;
    ls[j] = ns;
  }
  h2d(s.small4, sm.data(), sm.size() * sizeof(fe), st);
  msm_batch_on_device(g, vg, lg, kc, s.out, true);
  vdfgpu_gens gs = ipa_small_set(g->curve, s.pts, ns);
  msm_batch_on_device(&gs, vs, ls, kc, s.out + MSM_MAX_BATCH, true, false);
  fe* pin = pinned_evals();
  d2h(pin, s.out, kc * sizeof(jac_t), st);
  d2h(pin + 3 * MSM_MAX_BATCH, s.out + MSM_MAX_BATCH, kc * sizeof(jac_t), st);
  sync_after_unlock(st);
  copy_after_sync(out_host, pin, 2 * MSM_MAX_BATCH * sizeof(jac_t));
  normalise_after_sync(out_host, kc, g->curve);
  normalise_after_sync(reinterpret_cast<uint8_t*>(out_host) + MSM_MAX_BATCH * sizeof(jac_t), kc, g->curve);
}

// vdfgpu_ipa_verify_batch (ctx.cuh).  Like ipa_prove, the call holds a reference on g from its first guarded() section
// to its last; the batch is one section, each chunk of single-proof checks of a failing batch one more.  The verdicts
// fail closed: ok is zeroed first, and a 1 reaches it only when the whole call succeeded and that proof's check passed.
int ipa_verify_batch(vdfgpu_gens* g, size_t ell, size_t k, const IpaVerifyArgs& a, uint8_t* ok, const char* who,
                     IpaVerifyHook hook, void* hook_user) {
  IpaVerifyPlan p;
  IpaVerifyScratch s;
  bool holds_g = false;
  uint8_t sum[96];
  std::vector<uint8_t> verdict(k, 0);
  const std::string name(who);
  int rc = guarded([&] {
    if (!g || !a.comm || !a.a_hat || !a.c || !a.b_hat || !a.u_scale || !a.w || !ok || (ell && (!a.L || !a.R || !a.r)))
      throw ArgError(name + ": null pointer");   // L, R and r may be NULL at ell = 0
    if (k == 0) throw ArgError(name + ": no proofs");
    std::memset(ok, 0, k);
    if (ell > 40 || g->n < ((size_t)1 << ell) + 1)
      throw ArgError(name + ": the generator set needs at least 2^ell + 1 points");
    with_curve(g->curve, who, [&](auto C, auto BF, auto SF) {
      using F = decltype(SF);
      for (size_t i = 0; i < k * ell; i++)
        if (!usable_challenge<F>(a.r[i])) throw ArgError(name + ": a challenge is 0 or non-canonical");
      for (size_t q = 0; q < k; q++)
        if (!usable_challenge<F>(a.w[q])) throw ArgError(name + ": a weight is 0 or non-canonical");
      p = ipa_verify_prepare<decltype(BF), F>(ell, k, a);
      if (p.active.empty()) return;
      require_ready();
      g->refs++;
      holds_g = true;
      if (hook) hook(hook_user, p.active, cur_stream());
      ipa_verify_batch_enqueue<decltype(C), F>(g, ell, p, s, sum);
    });
  });
  const bool passed = rc == VDFGPU_OK && holds_g && std::all_of(sum + 64, sum + 96, [](uint8_t v) { return v == 0; });
  if (rc == VDFGPU_OK && holds_g && !passed) {
    for (size_t first = 0; rc == VDFGPU_OK && first < p.active.size(); first += MSM_MAX_BATCH) {
      const uint32_t kc = (uint32_t)std::min<size_t>(MSM_MAX_BATCH, p.active.size() - first);
      uint8_t res[2 * MSM_MAX_BATCH][96];
      rc = guarded([&] {
        require_ready();
        with_curve(g->curve, who, [&](auto, auto, auto SF) {
          ipa_verify_chunk_enqueue<decltype(SF)>(g, ell, p, s, first, kc, res);
        });
      });
      if (rc != VDFGPU_OK) break;
      // proof valid iff (its share over g) = -(its share over its own points): both normalised, identity all zero
      with_curve(g->curve, who, [&](auto, auto BF, auto) {
        using F = decltype(BF);
        for (uint32_t j = 0; j < kc; j++) {
          fe P[3], Q[3];
          std::memcpy(P, res[j], 96);
          std::memcpy(Q, res[MSM_MAX_BATCH + j], 96);
          verdict[p.active[first + j]] = F::eq(P[0], Q[0]) && F::eq(P[1], F::neg(Q[1])) && F::eq(P[2], Q[2]);
        }
      });
    }
  } else if (passed) {
    for (size_t q : p.active) verdict[q] = 1;
  }
  if (rc == VDFGPU_OK) std::memcpy(ok, verdict.data(), k);
  std::string keep = rc == VDFGPU_OK ? std::string() : std::string(vdfgpu_last_error());
  guarded([&] {
    if (holds_g) g->refs--;
    if (!ctx().ready) return;
    for (void* ptr : s.all())
      if (ptr) cudaFreeAsync(ptr, cur_stream());
  });
  if (rc != VDFGPU_OK) set_error(keep);
  return rc;
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

// ---- the inner-product argument on a resident generator set ----------------------------------------------------
int vdfgpu_ipa_prove(vdfgpu_gens* g, const void* a_host, const void* b_host, size_t ell, const void* u_scale32_host,
                     vdfgpu_ipa_round_fn round_fn, void* user, void* a_hat32_host) {
  return ipa_prove(g, const_cast<void*>(a_host), const_cast<void*>(b_host), true, ell, u_scale32_host, round_fn, user,
                   a_hat32_host);
}

int vdfgpu_ipa_prove_dev(vdfgpu_gens* g, void* a_dev, void* b_dev, size_t ell, const void* u_scale32_host,
                         vdfgpu_ipa_round_fn round_fn, void* user, void* a_hat32_host) {
  return ipa_prove(g, a_dev, b_dev, false, ell, u_scale32_host, round_fn, user, a_hat32_host);
}

int vdfgpu_ipa_gens_hat(vdfgpu_gens* g, const void* r_host, size_t ell, void* out_point96_host) {
  return guarded([&] {
    if (!g || !out_point96_host || (ell && !r_host)) throw ArgError("ipa_gens_hat: null pointer");
    if (ell > 40 || g->n < (size_t)1 << ell) throw ArgError("ipa_gens_hat: the generator set needs at least 2^ell points");
    std::vector<fe> r(ell ? ell : 1);
    if (ell) std::memcpy(r.data(), r_host, ell * sizeof(fe));
    std::vector<fe> r_inv(r.begin(), r.begin() + ell);
    with_curve(g->curve, "ipa_gens_hat", [&](auto, auto, auto SF) {
      for (size_t j = 0; j < ell; j++)
        if (!usable_challenge<decltype(SF)>(r[j])) throw ArgError("ipa_gens_hat: a challenge is 0 or non-canonical");
      batch_invert<decltype(SF)>(r_inv);
      require_ready();
      ipa_gens_hat_enqueue<decltype(SF)>(g, r.data(), r_inv.data(), ell, out_point96_host);
    });
  });
}

int vdfgpu_ipa_verify_batch(vdfgpu_gens* g, size_t ell, size_t k, const void* comm_a96_host, const void* L96_host,
                            const void* R96_host, const void* r32_host, const void* a_hat32_host, const void* c32_host,
                            const void* b_hat32_host, const void* u_scale32_host, const void* w32_host,
                            uint8_t* ok_out_host) {
  auto fes = [](const void* p) { return reinterpret_cast<const fe*>(p); };
  const IpaVerifyArgs a{reinterpret_cast<const uint8_t*>(comm_a96_host), reinterpret_cast<const uint8_t*>(L96_host),
                        reinterpret_cast<const uint8_t*>(R96_host), fes(r32_host), fes(a_hat32_host), fes(c32_host),
                        fes(b_hat32_host), fes(u_scale32_host), fes(w32_host), 1, 1, ell};
  return ipa_verify_batch(g, ell, k, a, ok_out_host, "ipa_verify_batch");
}

#pragma GCC visibility pop
}  // extern "C"
