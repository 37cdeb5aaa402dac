// Relaxed-R1CS kernels: sparse mat-vec (Az, Bz, Cz), fused folding cross-term T, and the fold update.
// They replace, inside nova-snark 0.8.0 (called from the reference at src/nova/proof.rs:342-349):
//   R1CSShape::multiply_vec      -> MultiplyVecFn       (SURVEY.md section 8a row a5)
//   R1CSShape::commit_T (T part) -> CrossTermFn         (row a6;  T = Az1.Bz2 + Az2.Bz1 - u1.Cz2 - u2.Cz1)
//   RelaxedR1CSWitness::fold     -> FoldFn              (row a7;  W <- W1 + r W2,  E <- E1 + r T)
//
// Layout in HBM: the three matrices are stored back to back as ONE CSR with 3*cons rows (A rows, then B,
// then C): row_ptr u32[3*cons+1], col u32[nnz], val 32-byte Montgomery field elements [nnz].  z is never
// materialised: column j < vars reads W[j], j == vars reads u, j > vars reads X[j-vars-1], so W stays
// resident across steps.  All kernels are bound by HBM bandwidth (36 B per non-zero + 32 B per row out).
#pragma once
#include "field.cuh"
#include "launch.cuh"

namespace vdf {

struct CsrView {
  const uint32_t* row_ptr;  // [3*cons + 1]
  const uint32_t* col;
  const fe* val;
  uint32_t cons, vars, io;
};

struct ZView {   // z = [W | u | X]
  const fe* W;
  const fe* u;   // one element
  const fe* X;
};

template <class F>
VDF_HD fe z_at(const ZView& z, uint32_t vars, uint32_t col) {
  const fe* p = col < vars ? z.W + col : (col == vars ? z.u : z.X + (col - vars - 1));
  return fe_load_gather(p);   // random 32-byte gather: do not pull the rest of the line
}

// acc += v * x.  Most R1CS coefficients are +1 or -1 (every A/B entry and all but one C entry of the MinRoot
// step circuit, src/nova/proof.rs:176-227): those cost an addition instead of a 245-instruction multiplication,
// which is what moves these kernels from the multiply pipe back to the HBM roofline.  Exact either way.
template <class F>
VDF_HD fe mul_acc(const fe& acc, const fe& v, const fe& x, const fe& one, const fe& minus_one) {
  if (F::eq(v, one)) return F::add(acc, x);
  if (F::eq(v, minus_one)) return F::sub(acc, x);
  return F::add(acc, F::mul(v, x));
}

template <class F>
VDF_HD fe csr_row_dot(const CsrView& m, uint32_t row, const ZView& z) {
  fe acc = F::zero();
  const fe one = F::one(), minus_one = F::neg(F::one());
  uint32_t lo = m.row_ptr[row], hi = m.row_ptr[row + 1];
  for (uint32_t k = lo; k < hi; k++) {
    fe v = fe_load(m.val + k);
    fe x = z_at<F>(z, m.vars, m.col[k]);
    acc = mul_acc<F>(acc, v, x, one, minus_one);
  }
  return acc;
}

// one thread per (matrix, row): out[mat][row]
template <class F>
struct MultiplyVecFn {
  CsrView m;
  ZView z;
  fe* Az; fe* Bz; fe* Cz;
  VDF_HD void operator()(size_t idx) const {
    uint32_t row = (uint32_t)idx;
    fe r = csr_row_dot<F>(m, row, z);
    uint32_t mat = row / m.cons, rr = row - mat * m.cons;
    fe* out = mat == 0 ? Az : (mat == 1 ? Bz : Cz);
    fe_store(out + rr, r);
  }
};

// one thread per constraint row: six dot products sharing the row's (col, val) loads, then
// T = Az1*Bz2 + Az2*Bz1 - u1*Cz2 - Cz1   (u2 = 1 for the fresh instance)
template <class F>
struct CrossTermFn {
  CsrView m;
  ZView z1, z2;
  fe* T;
  VDF_HD void operator()(size_t idx) const {
    uint32_t row = (uint32_t)idx;
    const fe one = F::one(), minus_one = F::neg(F::one());
    uint32_t ptr[3][2];
#pragma unroll
    for (uint32_t mat = 0; mat < 3; mat++) {   // six independent loads: one memory latency for all three matrices
      ptr[mat][0] = m.row_ptr[mat * m.cons + row];
      ptr[mat][1] = m.row_ptr[mat * m.cons + row + 1];
    }
    // (Measured and removed in round 2: prefetch.global.L2 of the later matrices' (col, val) entries and of the z
    // elements they select, issued here -- 0.245 -> 0.283 ms on the 2^21-constraint shape.  The kernel is not bound by
    // its chain of dependent loads: with full-size B coefficients a row costs 5 field multiplications for 252 bytes,
    // i.e. 0.14 ms of multiply pipe against 0.08 ms of HBM for this shape; see DESIGN.md section 2.3.)
    // the A and B products are combined as soon as both are known, so at most four dot products are live at once
    fe a1, a2, t;
#pragma unroll
    for (uint32_t mat = 0; mat < 3; mat++) {
      fe s1 = F::zero(), s2 = F::zero();
      uint32_t lo = ptr[mat][0], hi = ptr[mat][1];
      for (uint32_t k = lo; k < hi; k++) {
        fe v = fe_load(m.val + k);
        uint32_t c = m.col[k];
        s1 = mul_acc<F>(s1, v, z_at<F>(z1, m.vars, c), one, minus_one);
        s2 = mul_acc<F>(s2, v, z_at<F>(z2, m.vars, c), one, minus_one);
      }
      if (mat == 0) {
        a1 = s1; a2 = s2;
      } else if (mat == 1) {
        t = F::add(F::mul(a1, s2), F::mul(a2, s1));          // Az1*Bz2 + Az2*Bz1
      } else {
        t = F::sub(F::sub(t, F::mul(fe_load(z1.u), s2)), s1);   // - u1*Cz2 - Cz1
      }
    }
    fe_store(T + row, t);
  }
};

// ---- satisfiability: RelaxedR1CSShape::is_sat_relaxed / R1CSShape::is_sat [R], the row part of
// RecursiveSNARK::verify (src/nova/proof.rs:382) ------------------------------------------------------------------
// The two little-endian u64 counters of the C ABI (violating rows, smallest violating row), written as four u32
// words: RelaxedSatFn updates the low words (both values stay below 2^30) and only ever accesses them as u32.
struct SatInitFn {
  uint32_t* words;   // [4]
  uint32_t cons;
  VDF_HD void operator()(size_t) const {
    words[0] = 0; words[1] = 0;      // violating rows
    words[2] = cons; words[3] = 0;   // smallest violating row: cons = none
  }
};

// one thread per constraint row: d = Az*Bz - u*Cz - E[row] (E == nullptr: E = 0); the row violates the relation iff
// d != 0 (inputs are canonical, so zero has one encoding).  *bad counts the violating rows, *first ends as the smallest
// of them (it starts at cons).  Violations are rare in real use: one warp ballot, then lane 0 issues the atomics.
template <class F>
struct RelaxedSatFn {
  CsrView m;
  ZView z;
  const fe* E;
  uint32_t* bad;
  uint32_t* first;
  VDF_HD void operator()(size_t idx) const {
    const uint32_t row = (uint32_t)idx;
    const fe one = F::one(), minus_one = F::neg(F::one());
    uint32_t ptr[3][2];
#pragma unroll
    for (uint32_t mat = 0; mat < 3; mat++) {   // six independent loads, as in CrossTermFn
      ptr[mat][0] = m.row_ptr[mat * m.cons + row];
      ptr[mat][1] = m.row_ptr[mat * m.cons + row + 1];
    }
    fe d;   // Az, then Az*Bz, then the difference: one accumulator and one running value live at a time
#pragma unroll
    for (uint32_t mat = 0; mat < 3; mat++) {
      fe acc = F::zero();
      for (uint32_t k = ptr[mat][0]; k < ptr[mat][1]; k++)
        acc = mul_acc<F>(acc, fe_load(m.val + k), z_at<F>(z, m.vars, m.col[k]), one, minus_one);
      if (mat == 0) d = acc;
      else if (mat == 1) d = F::mul(d, acc);
      else d = F::sub(d, F::mul(fe_load(z.u), acc));
    }
    if (E) d = F::sub(d, fe_load(E + row));
    const bool violated = !F::eq(d, F::zero());
#if defined(__CUDA_ARCH__)
    // The lanes of this warp that hold a row: functor_kernel has already returned for i >= n, so the last warp is
    // partial when cons % 32 != 0.  The mask is computed from cons rather than taken from __activemask(): after the
    // data-dependent loops above the lanes need not have reconverged, and a ballot over a subset would lose counts.
    const uint32_t lane = threadIdx.x & 31u, base = row - lane;
    const uint32_t live = m.cons - base >= 32u ? 0xffffffffu : (1u << (m.cons - base)) - 1u;
    const uint32_t votes = __ballot_sync(live, violated);
    if (lane == 0 && votes) {
      atomic_add_u32(bad, (uint32_t)__popc(votes));
      atomic_min_u32(first, base + (uint32_t)(__ffs(votes) - 1));
    }
#else
    if (violated) {
      atomic_add_u32(bad, 1);
      atomic_min_u32(first, row);
    }
#endif
  }
};

// ---- transposed product for Spartan's inner sum-check (SURVEY 8f rank 2) ---------------------------------------
// M(y) = sum_x eq(x) * (rA A[x,y] + rB B[x,y] + rC C[x,y]) for every column y: nova-snark's
// compute_eval_table_sparse combined with the three challenges [R], reached from CompressedSNARK::prove
// (src/nova/proof.rs:363).  The scaled row table eq3[mat * cons + x] = r_mat * eq(x) first, then one THREAD per column
// over the column view (40 bytes per entry read in order + one gathered table element); the few heavy columns (the
// constant column of the step circuit holds one entry per round, with a full-size coefficient) are left to one BLOCK
// each: threads stride over the entries, shuffle trees and shared memory add them up.
struct CscView {
  const uint32_t* col_ptr;  // [ncols + 1]
  const uint32_t* srow;     // stacked row = mat * cons + row
  const fe* val;            // column order
  const uint32_t* heavy;    // columns with more than heavy_above entries
  uint32_t heavy_above;
};

template <class F>
struct ScaleRowsFn {
  const fe* eq;     // [cons]
  const fe* coef;   // [3]
  uint32_t cons;
  fe* eq3;          // [3 * cons]
  VDF_HD void operator()(size_t idx) const {
    const uint32_t mat = (uint32_t)(idx / cons), row = (uint32_t)(idx - (size_t)mat * cons);
    fe_store(eq3 + idx, F::mul(fe_load(coef + mat), fe_load(eq + row)));
  }
};

template <class F>
struct BindRowsFn {   // index = column
  CscView m;
  const fe* eq3;
  fe* out;          // [ncols]
  VDF_HD void operator()(size_t col) const {
    const uint32_t lo = m.col_ptr[col], hi = m.col_ptr[col + 1];
    if (hi - lo > m.heavy_above) return;   // BindHeavyFn's
    const fe one = F::one(), minus_one = F::neg(F::one());
    fe acc = F::zero();
    for (uint32_t k = lo; k < hi; k++)
      acc = mul_acc<F>(acc, fe_load(m.val + k), fe_load_gather(eq3 + m.srow[k]), one, minus_one);
    fe_store(out + col, acc);
  }
};

template <class F>
struct BindHeavyFn {   // index = (position in the heavy list) * THREADS + thread; launched with whole blocks of THREADS
  static constexpr uint32_t THREADS = 512;
  CscView m;
  const fe* eq3;
  fe* out;
  VDF_HD void operator()(size_t idx) const {
    const uint32_t col = m.heavy[idx / THREADS];
    const uint32_t lo = m.col_ptr[col], hi = m.col_ptr[col + 1];
    const fe one = F::one(), minus_one = F::neg(F::one());
    fe acc = F::zero();
#if defined(__CUDA_ARCH__)
    // the constant column of a t-round step circuit has ~3t entries with full-size coefficients: one multiplication
    // each, spread over the block; shuffle tree per warp, then the warp totals through shared memory
    __shared__ fe warp_tot[THREADS / 32];
    const unsigned tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    for (uint32_t k = lo + tid; k < hi; k += THREADS)
      acc = mul_acc<F>(acc, fe_load(m.val + k), fe_load_gather(eq3 + m.srow[k]), one, minus_one);
#pragma unroll 1
    for (int d = 16; d >= 1; d >>= 1) {
      fe o;
#pragma unroll
      for (int q = 0; q < 8; q++) o.v[q] = __shfl_down_sync(0xffffffffu, acc.v[q], d);
      acc = F::add(acc, o);
    }
    if (lane == 0) warp_tot[warp] = acc;
    __syncthreads();
    if (warp == 0) {
      acc = lane < THREADS / 32 ? warp_tot[lane] : F::zero();
#pragma unroll 1
      for (int d = 8; d >= 1; d >>= 1) {
        fe o;
#pragma unroll
        for (int q = 0; q < 8; q++) o.v[q] = __shfl_down_sync(0xffffffffu, acc.v[q], d);
        acc = F::add(acc, o);
      }
      if (lane == 0) fe_store(out + col, acc);
    }
#else
    if (idx % THREADS) return;
    for (uint32_t k = lo; k < hi; k++) acc = mul_acc<F>(acc, fe_load(m.val + k), fe_load(eq3 + m.srow[k]), one, minus_one);
    fe_store(out + col, acc);
#endif
  }
};

// ---- Spartan's padded layout (vdfgpu_running_spartan_prove, vdfgpu_r1cs_evaluate) -----------------------------
// nova's R1CSShape::pad [R]: m = the next power of two >= max(vars, cons); cons and vars are both padded to m, and the
// columns from u on move up by m - vars, so W occupies [0, m), u is column m and X starts at m + 1.  z then has 2m
// entries (ell_x = log2 m row variables, ell_y = ell_x + 1 column variables); 1 + io <= m is required.
struct PaddedLayout {
  uint32_t vars, io;
  size_t m;
  uint32_t ell_x;
  static PaddedLayout of(uint32_t cons, uint32_t vars, uint32_t io) {
    const uint32_t need = cons > vars ? cons : vars;
    uint32_t ell = 0;
    while (((size_t)1 << ell) < need) ell++;
    return PaddedLayout{vars, io, (size_t)1 << ell, ell};
  }
  bool fits() const { return 1 + (size_t)io <= m; }
  // padded column of the shape's column c
  VDF_HD size_t col(uint32_t c) const { return c < vars ? c : c + (m - vars); }
  // the shape's column at padded index j < 2m, or -1 for a padding slot (the inverse of col)
  VDF_HD int64_t source(size_t j) const {
    if (j < vars) return (int64_t)j;
    if (j < m || j > m + io) return -1;
    return (int64_t)(j - m + vars);
  }
  // a 2m-entry table over padded columns read through the shape's column numbers (z_at's mapping)
  VDF_HD ZView view(const fe* t) const { return ZView{t, t + m, t + m + 1}; }
};

// the outer sum-check's tables, one thread per padded row r < m: Az, Bz, Cz (RelaxedSatFn's row loop) and
// D = u Cz + E[r]; rows >= cons are zero.  E holds m entries (the zero-padded snapshot).
template <class F>
struct OuterTablesFn {
  CsrView m;
  ZView z;
  const fe* E;
  fe* Az; fe* Bz; fe* Cz; fe* D;
  VDF_HD void operator()(size_t idx) const {
    const uint32_t row = (uint32_t)idx;
    fe acc[3] = {F::zero(), F::zero(), F::zero()};
    if (row < m.cons) {
      const fe one = F::one(), minus_one = F::neg(F::one());
#pragma unroll
      for (uint32_t mat = 0; mat < 3; mat++) {
        const uint32_t lo = m.row_ptr[mat * m.cons + row], hi = m.row_ptr[mat * m.cons + row + 1];
        for (uint32_t k = lo; k < hi; k++)
          acc[mat] = mul_acc<F>(acc[mat], fe_load(m.val + k), z_at<F>(z, m.vars, m.col[k]), one, minus_one);
      }
    }
    fe_store(Az + idx, acc[0]);
    fe_store(Bz + idx, acc[1]);
    fe_store(Cz + idx, acc[2]);
    fe_store(D + idx, row < m.cons ? F::add(F::mul(fe_load(z.u), acc[2]), fe_load(E + idx)) : F::zero());
  }
};

// the inner sum-check's tables over 2m padded columns j: Mp[j] = M[source(j)], zp[j] = z[source(j)], 0 in padding slots.
// M: the bound rows (BindRowsFn's output over the shape's columns); z = [W | u | X] through z_at.
template <class F>
struct PaddedScatterFn {
  PaddedLayout pad;
  const fe* M;
  ZView z;
  fe* Mp; fe* zp;
  VDF_HD void operator()(size_t j) const {
    const int64_t c = pad.source(j);
    fe_store(Mp + j, c < 0 ? F::zero() : fe_load(M + c));
    fe_store(zp + j, c < 0 ? F::zero() : z_at<F>(z, pad.vars, (uint32_t)c));
  }
};

// ---- the sparse evaluation of k proofs in one pass (vdfgpu_r1cs_evaluate_batch, vdfgpu_spartan_verify_batch) ----------
// (A, B, C)(r_x,q, r_y,q) for q < k over the padded layout, sum over entries (x, c, v) of v eq(r_x,q)[x] eq(r_y,q)[col(c)].
// Per proof q, eq(r_x) and eq(r_y) are never written out: eq(r)[i] = Hi(r)[i >> lo_bits] Lo(r)[i & (2^lo_bits - 1)]
// (EqCombineFn's factorisation), lo_bits = floor(ell / 2).  Four half tables per proof, back to back at q * per:
// Hi(r_x), Lo(r_x), Hi(r_y), Lo(r_y) -- 2^9 entries each at ell_y = 18, about 4 MB at k = 64, resident in L2.
struct EqHalves {
  uint32_t bits[4];   // table t has 2^bits[t] entries: Hi(r_x), Lo(r_x), Hi(r_y), Lo(r_y)
  size_t off[4];      // its offset in a proof's record
  size_t per;         // entries per proof
  static EqHalves of(uint32_t ell_x) {
    const uint32_t ell_y = ell_x + 1;
    EqHalves h{{ell_x - ell_x / 2, ell_x / 2, ell_y - ell_y / 2, ell_y / 2}, {0, 0, 0, 0}, 0};
    for (int t = 0; t < 4; t++) {
      h.off[t] = h.per;
      h.per += (size_t)1 << h.bits[t];
    }
    return h;
  }
  // eq(r_x) (t = 0) or eq(r_y) (t = 2) of the proof whose record starts at `rec`, at index i: one multiplication
  template <class F>
  VDF_HD fe at(const fe* rec, int t, size_t i) const {
    return F::mul(fe_load(rec + off[t] + (i >> bits[t + 1])), fe_load(rec + off[t + 1] + (i & (((size_t)1 << bits[t + 1]) - 1))));
  }
};

// All k proofs' half tables in one launch, index space k per: entry e of table t of proof q is EqPartFn over the bit
// range of r that table covers (Hi: the first bits[0] / bits[2] coordinates, Lo: the rest).  rx: [k][ell_x],
// ry: [k][ell_x + 1], most significant variable first.
template <class F>
struct EqHalfTablesBatchFn {
  const fe* rx; const fe* ry;
  uint32_t ell_x;
  EqHalves h;
  fe* out;   // [k][h.per]
  VDF_HD void operator()(size_t idx) const {
    const size_t q = idx / h.per, e = idx - q * h.per;
    // which table: selects rather than a run-time index into h, which would put h in local memory
    const bool y = e >= h.off[2], lo = y ? e >= h.off[3] : e >= h.off[1];
    const size_t i = e - (y ? (lo ? h.off[3] : h.off[2]) : (lo ? h.off[1] : 0));
    const fe* r = y ? ry + q * (ell_x + 1) : rx + q * ell_x;
    const uint32_t hb = y ? h.bits[2] : h.bits[0], first = lo ? hb : 0u, nbits = lo ? (y ? h.bits[3] : h.bits[1]) : hb;
    const fe one = F::one();
    fe acc = one;
#pragma unroll 1
    for (uint32_t j = 0; j < nbits; j++) {
      const fe rj = fe_load(r + first + j);
      acc = F::mul(acc, ((i >> (nbits - 1 - j)) & 1u) ? rj : F::sub(one, rj));
    }
    fe_store(out + idx, acc);
  }
};

// One (row, proof) term of the batch: for row x < cons and proof q, acc[mat] += eq_x,q[x] sum_{entries (c, v) of row x
// of mat} v eq_y,q[col(c)].  One multiplication per entry for its eq_y value (from the halves), mul_acc's for v (an
// addition when v = +-1), four per row: nnz (1 + f) + 4 cons per proof, f the share of non-unit coefficients.
template <class F>
struct SparseEvalBatchFn {
  CsrView m;
  PaddedLayout pad;
  EqHalves h;
  const fe* tables;   // EqHalfTablesBatchFn's output, [k][h.per]
  size_t k;
  VDF_HD void add_row(fe (&acc)[3], size_t q, uint32_t row) const {
    const fe* rec = tables + q * h.per;
    const fe one = F::one(), minus_one = F::neg(F::one());
    const fe ex = h.at<F>(rec, 0, row);
#pragma unroll
    for (uint32_t mat = 0; mat < 3; mat++) {
      const uint32_t lo = m.row_ptr[mat * m.cons + row], hi = m.row_ptr[mat * m.cons + row + 1];
      fe s = F::zero();
      for (uint32_t e = lo; e < hi; e++)
        s = mul_acc<F>(s, fe_load(m.val + e), h.at<F>(rec, 2, pad.col(m.col[e])), one, minus_one);
      acc[mat] = F::add(acc[mat], F::mul(ex, s));
    }
  }
};

#if defined(__CUDACC__)
constexpr int SE_BLOCK = 256;

// SparseEvalBatchFn over all rows and proofs.  Proofs fastest: the kq = 2^kq_log lanes of a group (kq = k rounded up
// to a power of two, at most 32) take the proofs blockIdx.y kq + lane, the 32 / kq groups of a warp take different
// rows, so at k >= 32 a warp's row_ptr, col and val loads are broadcasts.  Each thread runs a strided loop over rows
// with its proof fixed and three accumulators; a block's sums go to partial[(blockIdx.x k + q) 3 + mat]
// (sc_column_sum_kernel adds them up over gridDim.x blocks).
template <class F>
__global__ void __launch_bounds__(SE_BLOCK) sparse_eval_batch_kernel(const SparseEvalBatchFn<F> f, uint32_t kq_log,
                                                                     fe* partial) {
  const uint32_t kq = 1u << kq_log, lane_q = threadIdx.x & (kq - 1u), rows_per_block = SE_BLOCK >> kq_log;
  const size_t q = (size_t)blockIdx.y * kq + lane_q;
  fe acc[3] = {F::zero(), F::zero(), F::zero()};
  if (q < f.k)
    for (size_t row = (size_t)blockIdx.x * rows_per_block + (threadIdx.x >> kq_log); row < f.m.cons;
         row += (size_t)gridDim.x * rows_per_block)
      f.add_row(acc, q, (uint32_t)row);
  // the lanes of one proof in a warp differ in the bits above kq_log: a butterfly over those bits
#pragma unroll 1
  for (uint32_t d = 16; d >= kq; d >>= 1)
#pragma unroll
    for (int mat = 0; mat < 3; mat++) {
      fe o;
#pragma unroll
      for (int w = 0; w < 8; w++) o.v[w] = __shfl_xor_sync(0xffffffffu, acc[mat].v[w], d);
      acc[mat] = F::add(acc[mat], o);
    }
  __shared__ fe sm[3][SE_BLOCK / 32][32];
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  if (lane < kq)
#pragma unroll
    for (int mat = 0; mat < 3; mat++) sm[mat][warp][lane] = acc[mat];
  __syncthreads();
  if (threadIdx.x < 3 * kq) {
    const uint32_t mat = threadIdx.x >> kq_log, ql = threadIdx.x & (kq - 1u);
    fe s = sm[mat][0][ql];
#pragma unroll 1
    for (int w = 1; w < SE_BLOCK / 32; w++) s = F::add(s, sm[mat][w][ql]);
    const size_t qq = (size_t)blockIdx.y * kq + ql;
    if (qq < f.k) fe_store(partial + ((size_t)blockIdx.x * f.k + qq) * 3 + mat, s);
  }
}
#endif  // __CUDACC__

// a[i] <- a[i] + r * b[i] over two vectors in one launch (W with W2, E with T)
template <class F>
struct FoldFn {
  fe* W1; const fe* W2; size_t nW;
  fe* E1; const fe* T; size_t nE;
  const fe* r;
  VDF_HD void operator()(size_t i) const {
    fe rr = fe_load(r);
    if (i < nW) {
      fe_store(W1 + i, F::add(fe_load(W1 + i), F::mul(rr, fe_load(W2 + i))));
    } else {
      size_t j = i - nW;
      fe_store(E1 + j, F::add(fe_load(E1 + j), F::mul(rr, fe_load(T + j))));
    }
  }
};

}  // namespace vdf
