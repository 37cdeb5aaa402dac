// Sum-check building blocks over multilinear polynomials in evaluation form (tables of 2^k field elements):
// what CompressedSNARK::prove (reference src/nova/proof.rs:360-368) spends its non-MSM time in, inside nova-snark
// 0.8's spartan_with_ipa_pc (SURVEY.md section 8f rank 2).  [R]: that crate is not under /root/reference; the
// semantics below restate its sumcheck.rs / polynomial.rs from memory and are unique mathematical objects:
//
//   EqPolynomial::evals            eq[idx] = prod_j (bit_j(idx) ? r_j : 1 - r_j), r_0 <-> most significant bit
//   prove_cubic_with_additive_term one round: (e0, e2, e3) = sum_i comb(P(0), ..), comb(P(2), ..), comb(P(3), ..) with
//                                  comb(A, B, C, D) = A (B C - D), P(0) = lo, P(2) = 2 hi - lo, P(3) = 3 hi - 2 lo,
//                                  lo = P[i], hi = P[i + len/2]   (outer sum-check: A = eq(tau), B = Az, C = Bz, D = u Cz + E)
//   prove_quad                     one round: (e0, e2) with comb(A, B) = A B  (inner sum-check: ABC(r_x, .) and z)
//   bound_poly_var_top             P[i] <- lo + r (hi - lo), length halves
//   MultilinearPolynomial::evaluate  = <eq(r), P>
//
// All of it is streaming work over tables: 32 B per element read once per round -- HBM-bound at large sizes (the
// cubic round does 6 multiplications per 256 bytes: about even between the multiply pipe and HBM), launch-bound at
// Nova's own sizes (2^14 - 2^17 entries, L2-resident).  Reductions: per-thread strided partial sums, a shuffle tree
// per warp, shared memory across the warps of a block, one partial per block, a second one-block launch.
#pragma once
#include "curve.cuh"
#include "field.cuh"
#include "launch.cuh"

namespace vdf {

// ---- inner-product-argument building blocks (the polynomial-commitment opening of spartan_with_ipa_pc, [R]) --------
// One IPA round halves the vectors and the generators with the challenge r:
//   a' = r a_L + r^-1 a_R,  b' = r^-1 b_L + r b_R              (VecLinCombFn: out[i] = x a[i] + y b[i])
//   G'_i = r^-1 G_L,i + r G_R,i   (CommitGens::fold: n/2 independent two-term scalar multiplications;
//                                  nova computes each with vartime_multiscalar_mul on two points)
//   c_L = <a_L, b_R>, c_R = <a_R, b_L>                        (sc_dot_kernel below)
template <class F>
struct VecLinCombFn {
  const fe* a; const fe* b; const fe* xy;   // xy[0] = x, xy[1] = y (Montgomery)
  fe* out;
  VDF_HD void operator()(size_t i) const {
    fe_store(out + i, F::add(F::mul(fe_load(xy), fe_load(a + i)), F::mul(fe_load(xy + 1), fe_load(b + i))));
  }
};

// out[i] = w1 P[i] + w2 Q[i] on packed affine points, normalised to affine again.  Thread = CH consecutive outputs:
// each by interleaved double-and-add over the bits of both scalars (Shamir's trick: one doubling per bit, one addition
// of P, Q or P + Q), then ONE inversion for the CH results (Montgomery's trick).  C = curve, SF = its scalar field.
template <class C, class F, class SF>
struct PointLinCombFn {
  const affine_t* P; const affine_t* Q;
  const fe* w;            // w[0] = w1, w[1] = w2 (Montgomery, scalar field)
  affine_t* out;
  size_t n;
  static constexpr int CH = 4;
  VDF_HD void operator()(size_t t) const {
    const size_t lo = t * CH, hi = lo + CH < n ? lo + CH : n;
    const fe k1 = SF::from_mont(fe_load(w)), k2 = SF::from_mont(fe_load(w + 1));
    xyzz_t res[CH];
    fe pref[CH];
    fe run = F::one();
    for (size_t i = lo; i < hi; i++) {
      affine_t p, q;
      p.x = fe_load(&P[i].x); p.y = fe_load(&P[i].y);
      q.x = fe_load(&Q[i].x); q.y = fe_load(&Q[i].y);
      xyzz_t pq = C::from_affine(p);
      C::madd_signed(pq, q, false);                       // P + Q (identity operands and P = +-Q handled inside)
      xyzz_t acc = C::identity();
#pragma unroll 1
      for (int bit = 255; bit >= 0; bit--) {
        acc = C::dbl(acc);
        const uint32_t b1 = (k1.v[bit >> 5] >> (bit & 31)) & 1u, b2 = (k2.v[bit >> 5] >> (bit & 31)) & 1u;
        if (b1 & b2) C::add(acc, pq);
        else if (b1) C::madd_signed(acc, p, false);
        else if (b2) C::madd_signed(acc, q, false);
      }
      res[i - lo] = acc;
      pref[i - lo] = run;
      if (!C::is_inf(acc)) run = F::mul(run, F::mul(acc.ZZ, acc.ZZZ));
    }
    fe inv = F::inv(run);
    for (size_t i = hi; i > lo; i--) {
      const xyzz_t& r = res[i - 1 - lo];
      affine_t a;
      if (C::is_inf(r)) {
        a.x = F::zero(); a.y = F::zero();
      } else {
        const fe zi = F::mul(inv, pref[i - 1 - lo]);        // 1 / (ZZ * ZZZ)
        inv = F::mul(inv, F::mul(r.ZZ, r.ZZZ));
        a.x = F::mul(r.X, F::mul(zi, r.ZZZ));
        a.y = F::mul(r.Y, F::mul(zi, r.ZZ));
      }
      fe_store(&out[i - 1].x, a.x);
      fe_store(&out[i - 1].y, a.y);
    }
  }
};

// ---- the whole inner-product argument on a resident generator set (vdfgpu_ipa_prove, vdfgpu_ipa_gens_hat) ----------
// n = 2^ell; a, b in the scalar field of g's curve (Montgomery); g holds at least n + 1 points, G_k = point k, and
// U0 = G_n is nova's gens_c; U = u_scale U0 (nova scales gens_c by a transcript scalar first, gens_c.scale(&r) [R]).
// Round j = 0 .. ell-1, m = n / 2^j, h = m / 2:
//   c_L = <a[0,h), b[h,m)>,  c_R = <a[h,m), b[0,h)>
//   L = <a[0,h), G'[h,m)> + c_L U,  R = <a[h,m), G'[0,h)> + c_R U;  the caller's transcript turns (L, R) into r != 0
//   a <- r a_L + r^-1 a_R,  b <- r^-1 b_L + r b_R,  G' <- r^-1 G'_L + r G'_R;   a_hat = a[0] after ell rounds.
// s_k = prod_j (bit_j(k) ? r_j : r_j^-1), bit_0 the most significant of the ell bits (nova's s), G_hat = <s, G[0,n)>.
// The generators are never folded: G'_j[i] = sum_t coef_j[t] G[t m + i] with coef_0 = [1],
// coef_{j+1}[2t + beta] = coef_j[t] (beta ? r_j : r_j^-1), so coef_ell = s, and L and R are ONE batched MSM over the
// original resident set with the scalars IpaExpandFn writes.  Folding n points per round instead is a 256-bit
// double-and-add per output (PointLinCombFn, ~4 500 multiplications each) plus a plain-layout MSM per round.

// Round j's commitment scalars over G[0, n], k = t m + i (i < m, m = 2^log_m, h = m / 2), index space n + 1:
//   SL[k] = a[i - h] coef[t] if i >= h else 0,  SR[k] = a[i + h] coef[t] if i < h else 0,
//   SL[n] = c[0] u_scale,  SR[n] = c[1] u_scale       (c = (c_L, c_R), on the device)
template <class F>
struct IpaExpandFn {
  const fe* a; const fe* coef; const fe* c;
  fe u_scale;
  uint32_t log_m;
  size_t n;
  fe* SL; fe* SR;
  VDF_HD void operator()(size_t k) const {
    if (k == n) {
      fe_store(SL + n, F::mul(fe_load(c), u_scale));
      fe_store(SR + n, F::mul(fe_load(c + 1), u_scale));
      return;
    }
    const size_t h = (size_t)1 << (log_m - 1), i = k & ((h << 1) - 1);
    const bool left = i < h;
    const fe v = F::mul(fe_load(a + (left ? i + h : i - h)), fe_load(coef + (k >> log_m)));
    fe_store(SL + k, left ? F::zero() : v);
    fe_store(SR + k, left ? v : F::zero());
  }
};

// The fold of one round, index space max(h, nc):
//   a[i] <- r a[i] + r^-1 a[h + i],  b[i] <- r^-1 b[i] + r b[h + i]        for i < h (in place)
//   coef_out[2t] = coef_in[t] r^-1,  coef_out[2t + 1] = coef_in[t] r      for t < nc
// With h = 0 it only doubles coef (the s table of vdfgpu_ipa_gens_hat).
template <class F>
struct IpaFoldFn {
  fe* a; fe* b;
  size_t h;
  const fe* coef_in; fe* coef_out;
  size_t nc;
  fe r, r_inv;
  VDF_HD void operator()(size_t i) const {
    if (i < h) {
      fe_store(a + i, F::add(F::mul(r, fe_load(a + i)), F::mul(r_inv, fe_load(a + h + i))));
      fe_store(b + i, F::add(F::mul(r_inv, fe_load(b + i)), F::mul(r, fe_load(b + h + i))));
    }
    if (i < nc) {
      const fe c = fe_load(coef_in + i);
      fe_store(coef_out + 2 * i, F::mul(c, r_inv));
      fe_store(coef_out + 2 * i + 1, F::mul(c, r));
    }
  }
};

// ---- batch verification of inner-product arguments (vdfgpu_ipa_verify_batch) -------------------------------------
// Proof q (of k) over the same set is valid iff
//   a_hat G_hat + u_scale (a_hat b_hat - c) U0 - comm_a - sum_j (r_j^2 L_j + r_j^-2 R_j) = O,   G_hat = <s_q, G[0,n)>
// (ipa_ref.verify with P = comm_a + c U).  The equation is linear in the points, so with weights w_q != 0 the batch
// checks the weighted sum of the k left-hand sides with two MSMs:
//   over G[0, n]:            S[i] = sum_q w_q a_hat_q s_q[i]  (i < n),   S[n] = sum_q w_q u_scale_q (a_hat_q b_hat_q - c_q)
//   over the proofs' points: -w_q for comm_a_q, -w_q r_qj^2 for L_qj, -w_q r_qj^-2 for R_qj.
// S is built without k s tables: with ell_h = ceil(ell / 2) high bits and ell_l = floor(ell / 2) low bits of the index,
// s_q[t 2^ell_l + u] = Hi_q[t] Lo_q[u] (Hi over r_0 .. r_{ell_h - 1}, Lo over the rest), so S = sum_q Hi_q[t] Lo_q[u]
// is a field "matrix product" with inner dimension k: k multiplications per entry, from two tables of k 2^ell_h
// entries each at most (4 MB at k = 64, ell = 20), which stay in L2.

// All k Hi tables, then all k Lo tables, index space k (2^hi_bits + 2^lo_bits), hi_bits = ell - lo_bits:
//   hi[q 2^hi_bits + t] = scale[q] prod_{j < hi_bits} (bit_j(t) ? r[q][j] : r_inv[q][j])
//   lo[q 2^lo_bits + u] =          prod_{j < lo_bits} (bit_j(u) ? r[q][hi_bits + j] : r_inv[q][hi_bits + j])
// bit_0 the most significant; r and r_inv are [k][ell], proof-major.  scale = w a_hat (batch) or a_hat (one proof).
template <class F>
struct IpaHalfTablesFn {
  const fe* r; const fe* r_inv; const fe* scale;
  uint32_t ell, lo_bits;
  size_t k;
  fe* hi; fe* lo;
  VDF_HD void operator()(size_t idx) const {
    const uint32_t hi_bits = ell - lo_bits;
    const size_t hi_len = k << hi_bits;
    const bool is_hi = idx < hi_len;
    const size_t e = is_hi ? idx : idx - hi_len;
    const uint32_t nbits = is_hi ? hi_bits : lo_bits, first = is_hi ? 0u : hi_bits;
    const size_t q = e >> nbits, t = e & (((size_t)1 << nbits) - 1);
    fe acc = is_hi ? fe_load(scale + q) : F::one();
    const fe* rq = r + q * ell + first;
    const fe* riq = r_inv + q * ell + first;
#pragma unroll 1
    for (uint32_t j = 0; j < nbits; j++)
      acc = F::mul(acc, fe_load(((t >> (nbits - 1 - j)) & 1u) ? rq + j : riq + j));
    fe_store((is_hi ? hi : lo) + e, acc);
  }
};

// S[t 2^lo_bits + u] = sum_{q < k} hi[q 2^hi_bits + t] lo[q 2^lo_bits + u], S[n] = last (n = 2^(hi_bits + lo_bits)),
// index space n + 1.  Adjacent threads take adjacent u: the warp reads lo coalesced and hi as a broadcast.
template <class F>
struct IpaBatchScalarsFn {
  const fe* hi; const fe* lo;
  uint32_t hi_bits, lo_bits;
  size_t k;
  fe last;
  fe* S;
  VDF_HD void operator()(size_t i) const {
    const size_t n = (size_t)1 << (hi_bits + lo_bits);
    if (i == n) {
      fe_store(S + n, last);
      return;
    }
    const size_t t = i >> lo_bits, u = i & (((size_t)1 << lo_bits) - 1);
    const fe* h = hi + t;
    const fe* l = lo + u;
    fe acc = F::mul(fe_load(h), fe_load(l));
#pragma unroll 1
    for (size_t q = 1; q < k; q++) {
      h += (size_t)1 << hi_bits;
      l += (size_t)1 << lo_bits;
      acc = F::add(acc, F::mul(fe_load(h), fe_load(l)));
    }
    fe_store(S + i, acc);
  }
};

// ---- Spartan over a resident running instance (vdfgpu_running_spartan_prove) ---------------------------------------
// RelaxedR1CSSNARK::prove [R] on the padded layout (r1cs.cuh PaddedLayout; m rows, 2m columns, ell_x = log2 m):
//   outer  sum_x eq(tau, x) (Az(x) Bz(x) - (u Cz(x) + E(x))) = 0, cubic sum-check over ell_x rounds -> r_x,
//          claim_Az, claim_Bz from the bound tables, claim_Cz = <Cz, eq(r_x)>, eval_E = <E, eq(r_x)>
//   inner  sum_y M(y) z(y) = r_A claim_Az + r_B claim_Bz + r_C claim_Cz with M(y) = sum_x eq(r_x, x) (r_A A + r_B B +
//          r_C C)[x, y], quadratic sum-check over ell_x + 1 rounds -> r_y;  r_y' = r_y[1..]
//   claims eval_W = <W, eq(r_y')>; the two evaluation claims E(r_x) = eval_E and W(r_y') = eval_W are folded into one
//          inner-product claim with the challenge rho (nova's fold of two inner-product instances [R]):
//          T = <E, eq(r_y')> + <W, eq(r_x)>,  a = E + rho W,  b = eq(r_x) + rho eq(r_y'),
//          c = eval_E + rho T + rho^2 eval_W   (= <a, b>; its commitment is comm_E + rho comm_W)
//   open   the inner-product argument of <a, b> = c (vdfgpu_ipa_prove above).

// K inner products in one pass: out[q] = sum_{i < len[q]} v[q][i] eq[q][i].  Every vector may be shorter than the
// launch's n entries: the entries past len[q] are zero (implicit padding, nothing is read there).
template <int K>
struct MultiDot {
  const fe* v[K];
  const fe* eq[K];
  size_t len[K];
  template <class F>
  VDF_HD void add_terms(fe (&acc)[K], size_t i) const {
#pragma unroll
    for (int q = 0; q < K; q++)
      if (i < len[q]) acc[q] = F::add(acc[q], F::mul(fe_load(v[q] + i), fe_load(eq[q] + i)));
  }
};

// a[i] = E[i] + rho W[i], b[i] = eqx[i] + rho eqy[i]: the joint inner-product claim's vectors (a may be E, b may be eqx)
template <class F>
struct IpaJoinFn {
  const fe* E; const fe* W; const fe* eqx; const fe* eqy;
  fe rho;
  fe* a; fe* b;
  VDF_HD void operator()(size_t i) const {
    const fe e = fe_load(E + i), w = fe_load(W + i), x = fe_load(eqx + i), y = fe_load(eqy + i);
    fe_store(a + i, F::add(e, F::mul(rho, w)));
    fe_store(b + i, F::add(x, F::mul(rho, y)));
  }
};

constexpr int SC_BLOCK = 256;
constexpr int SC_MAX_POLYS = 4;

struct PolySet {
  fe* p[SC_MAX_POLYS];
};

// eq table over the bit range [first, first + nbits) of r (most significant first): out[idx], idx < 2^nbits
template <class F>
struct EqPartFn {
  const fe* r;       // [ell] Montgomery
  uint32_t first, nbits;
  fe* out;
  VDF_HD void operator()(size_t idx) const {
    fe acc = F::one();
    const fe one = F::one();
    for (uint32_t j = 0; j < nbits; j++) {
      const fe rj = fe_load(r + first + j);
      const bool bit = (idx >> (nbits - 1 - j)) & 1u;
      acc = F::mul(acc, bit ? rj : F::sub(one, rj));
    }
    fe_store(out + idx, acc);
  }
};

// out[idx] = hi[idx >> lo_bits] * lo[idx & (2^lo_bits - 1)]: one multiplication and one 32-byte store per entry
template <class F>
struct EqCombineFn {
  const fe* hi;
  const fe* lo;
  uint32_t lo_bits;
  fe* out;
  VDF_HD void operator()(size_t idx) const {
    fe_store(out + idx, F::mul(fe_load(hi + (idx >> lo_bits)), fe_load(lo + (idx & (((size_t)1 << lo_bits) - 1)))));
  }
};

// P[i] <- P[i] + r (P[i + half] - P[i]) for i < half, k polynomials in one launch (index = poly * half + i)
template <class F>
struct BindTopFn {
  PolySet polys;
  size_t half;
  const fe* r;
  VDF_HD void operator()(size_t idx) const {
    const size_t q = idx / half, i = idx - q * half;
    fe* P = polys.p[q];
    const fe lo = fe_load(P + i), hi = fe_load(P + half + i);
    fe_store(P + i, F::add(lo, F::mul(fe_load(r), F::sub(hi, lo))));
  }
};

// BindTopFn with the challenge as a kernel argument: the round loop has it on the host, one upload fewer per round
template <class F>
struct BindTopValFn {
  PolySet polys;
  size_t half;
  fe r;
  VDF_HD void operator()(size_t idx) const {
    const size_t q = idx / half, i = idx - q * half;
    fe* P = polys.p[q];
    const fe lo = fe_load(P + i), hi = fe_load(P + half + i);
    fe_store(P + i, F::add(lo, F::mul(r, F::sub(hi, lo))));
  }
};

#if defined(__CUDACC__)
// ---- reductions ------------------------------------------------------------------------------------------
template <class F>
__device__ __forceinline__ fe warp_sum(fe v) {
#pragma unroll 1
  for (int d = 16; d >= 1; d >>= 1) {
    fe o;
#pragma unroll
    for (int k = 0; k < 8; k++) o.v[k] = __shfl_down_sync(0xffffffffu, v.v[k], d);
    v = F::add(v, o);
  }
  return v;
}

// block-wide sums of NACC per-thread accumulators -> out[blockIdx.x * NACC + a]
template <class F, int NACC>
__device__ __forceinline__ void block_sum_store(fe (&acc)[NACC], fe* out) {
  __shared__ fe sm[NACC][SC_BLOCK / 32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int a = 0; a < NACC; a++) {
    fe s = warp_sum<F>(acc[a]);
    if (lane == 0) sm[a][wid] = s;
  }
  __syncthreads();
  if (wid == 0) {
#pragma unroll
    for (int a = 0; a < NACC; a++) {
      fe s = lane < SC_BLOCK / 32 ? sm[a][lane] : F::zero();
      s = warp_sum<F>(s);
      if (lane == 0) fe_store(out + (size_t)blockIdx.x * NACC + a, s);
    }
  }
}

// one round of the cubic sum-check with additive term: per-block partials of (e0, e2, e3)
template <class F>
__global__ void __launch_bounds__(SC_BLOCK) sc_cubic_round_kernel(const fe* A, const fe* B, const fe* C, const fe* D,
                                                                   size_t half, fe* partial) {
  fe acc[3] = {F::zero(), F::zero(), F::zero()};
  for (size_t i = (size_t)blockIdx.x * SC_BLOCK + threadIdx.x; i < half; i += (size_t)gridDim.x * SC_BLOCK) {
    fe a = fe_load(A + i), b = fe_load(B + i), c = fe_load(C + i), d = fe_load(D + i);
    acc[0] = F::add(acc[0], F::mul(a, F::sub(F::mul(b, c), d)));
    const fe ah = fe_load(A + half + i), bh = fe_load(B + half + i), ch = fe_load(C + half + i), dh = fe_load(D + half + i);
    const fe da = F::sub(ah, a), db = F::sub(bh, b), dc = F::sub(ch, c), dd = F::sub(dh, d);
    a = F::add(ah, da); b = F::add(bh, db); c = F::add(ch, dc); d = F::add(dh, dd);          // P(2) = 2 hi - lo
    acc[1] = F::add(acc[1], F::mul(a, F::sub(F::mul(b, c), d)));
    a = F::add(a, da); b = F::add(b, db); c = F::add(c, dc); d = F::add(d, dd);              // P(3) = P(2) + hi - lo
    acc[2] = F::add(acc[2], F::mul(a, F::sub(F::mul(b, c), d)));
  }
  block_sum_store<F, 3>(acc, partial);
}

// one round of the quadratic sum-check: per-block partials of (e0, e2)
template <class F>
__global__ void __launch_bounds__(SC_BLOCK) sc_quad_round_kernel(const fe* A, const fe* B, size_t half, fe* partial) {
  fe acc[2] = {F::zero(), F::zero()};
  for (size_t i = (size_t)blockIdx.x * SC_BLOCK + threadIdx.x; i < half; i += (size_t)gridDim.x * SC_BLOCK) {
    const fe a = fe_load(A + i), b = fe_load(B + i), ah = fe_load(A + half + i), bh = fe_load(B + half + i);
    acc[0] = F::add(acc[0], F::mul(a, b));
    acc[1] = F::add(acc[1], F::mul(F::add(ah, F::sub(ah, a)), F::add(bh, F::sub(bh, b))));
  }
  block_sum_store<F, 2>(acc, partial);
}

// <a, b> over n entries: per-block partials
template <class F>
__global__ void __launch_bounds__(SC_BLOCK) sc_dot_kernel(const fe* A, const fe* B, size_t n, fe* partial) {
  fe acc[1] = {F::zero()};
  for (size_t i = (size_t)blockIdx.x * SC_BLOCK + threadIdx.x; i < n; i += (size_t)gridDim.x * SC_BLOCK)
    acc[0] = F::add(acc[0], F::mul(fe_load(A + i), fe_load(B + i)));
  block_sum_store<F, 1>(acc, partial);
}

// (<A[0,h), B[h,2h)>, <A[h,2h), B[0,h)>), the IPA's (c_L, c_R): per-block partials
template <class F>
__global__ void __launch_bounds__(SC_BLOCK) sc_cross_dot_kernel(const fe* A, const fe* B, size_t half, fe* partial) {
  fe acc[2] = {F::zero(), F::zero()};
  for (size_t i = (size_t)blockIdx.x * SC_BLOCK + threadIdx.x; i < half; i += (size_t)gridDim.x * SC_BLOCK) {
    acc[0] = F::add(acc[0], F::mul(fe_load(A + i), fe_load(B + half + i)));
    acc[1] = F::add(acc[1], F::mul(fe_load(A + half + i), fe_load(B + i)));
  }
  block_sum_store<F, 2>(acc, partial);
}

// K inner products over n entries (MultiDot above): per-block partials
template <class F, int K>
__global__ void __launch_bounds__(SC_BLOCK) sc_multi_dot_kernel(const MultiDot<K> d, size_t n, fe* partial) {
  fe acc[K];
#pragma unroll
  for (int q = 0; q < K; q++) acc[q] = F::zero();
  for (size_t i = (size_t)blockIdx.x * SC_BLOCK + threadIdx.x; i < n; i += (size_t)gridDim.x * SC_BLOCK)
    d.template add_terms<F>(acc, i);
  block_sum_store<F, K>(acc, partial);
}

// second stage: out[a] = sum over blocks of partial[block * NACC + a]; one block
template <class F, int NACC>
__global__ void __launch_bounds__(SC_BLOCK) sc_final_kernel(const fe* partial, uint32_t nblocks, fe* out) {
  fe acc[NACC];
#pragma unroll
  for (int a = 0; a < NACC; a++) acc[a] = F::zero();
  for (uint32_t b = threadIdx.x; b < nblocks; b += SC_BLOCK)
#pragma unroll
    for (int a = 0; a < NACC; a++) acc[a] = F::add(acc[a], fe_load(partial + (size_t)b * NACC + a));
  block_sum_store<F, NACC>(acc, out);   // gridDim.x == 1: writes out[0 .. NACC)
}

// second stage of a reduction with many outputs: out[o] = sum over blocks b of partial[b * n_out + o]; one block per
// output (gridDim.x == n_out)
template <class F>
__global__ void __launch_bounds__(SC_BLOCK) sc_column_sum_kernel(const fe* partial, uint32_t nblocks, size_t n_out,
                                                                 fe* out) {
  fe acc[1] = {F::zero()};
  for (uint32_t b = threadIdx.x; b < nblocks; b += SC_BLOCK)
    acc[0] = F::add(acc[0], fe_load(partial + (size_t)b * n_out + blockIdx.x));
  block_sum_store<F, 1>(acc, out);   // writes out[blockIdx.x]
}

// grid for a reduction over `items`: enough blocks to fill the GPU, never more partials than the final block likes
static inline uint32_t sc_grid(size_t items) {
  size_t blocks = (items + SC_BLOCK - 1) / SC_BLOCK;
  const size_t cap = 148 * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (uint32_t)blocks;
}
#endif  // __CUDACC__

}  // namespace vdf
