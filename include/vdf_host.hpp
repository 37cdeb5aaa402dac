// vdf_host.hpp -- header-only C++17 host layer over the C ABI (vdfgpu.h), mirroring the names and argument
// meaning of the reference's Rust interfaces for the hot path so that a port of its call sites reads the same:
//
//   src/minroot.rs   State<T> (:267-272), trait MinRootVDF { check, inverse_eval, element, inverse_exponent }
//                    (:287-374), PallasVDF (:40), VestaVDF (:201), Evaluation { result, t, verify, append } (:376-439)
//   nova-snark 0.8   CommitGens / commit() -> Group::vartime_multiscalar_mul, R1CSShape::{multiply_vec, commit_T},
//                    RelaxedR1CSWitness::fold, NIFS::prove's witness side (reached from src/nova/proof.rs:342-349)
//
// Field elements and points are passed as the byte images pasta_curves (feature repr-c) keeps in memory:
// Fe = 32 bytes (4 x u64 LE, Montgomery), Affine = 72 bytes, Point = 96 bytes (Jacobian; results normalised).
// Errors: the infallible hooks of the reference (MSM, check) throw std::runtime_error where Rust would panic.
// There is no CPU fallback: every call needs libvdfgpu.so and a B200.
#pragma once
#include <array>
#include <cstdint>
#include <cstring>
#include <initializer_list>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

#include "vdfgpu.h"

namespace vdf_host {

using Fe = std::array<uint8_t, 32>;
using Affine = std::array<uint8_t, 72>;
using Point = std::array<uint8_t, 96>;

inline void ok_or_throw(int rc, const char* what) {
  if (rc != VDFGPU_OK) throw std::runtime_error(std::string(what) + ": " + vdfgpu_last_error());
}

inline void init(int device = 0) { ok_or_throw(vdfgpu_init(device), "vdfgpu_init"); }

// ---- src/minroot.rs ----------------------------------------------------------------------------------
struct State {  // State<G::Scalar>, minroot.rs:267-272; repr(C): x, y, i
  Fe x, y, i;
  bool operator==(const State& o) const { return x == o.x && y == o.y && i == o.i; }
};
static_assert(sizeof(State) == 96, "State must be three packed field elements");

template <int FIELD>
struct MinRootVDF {  // the fast direction of trait MinRootVDF<G>, minroot.rs:287-374
  static constexpr uint64_t inverse_exponent() { return 5; }  // minroot.rs:68-70, :215-217

  // check(result, t, original) for many independent triples (minroot.rs:369-371)
  static std::vector<bool> check_batch(const std::vector<State>& results, const std::vector<uint64_t>& t,
                                       const std::vector<State>& originals) {
    if (results.size() != originals.size() || (t.size() != results.size() && t.size() != 1))
      throw std::invalid_argument("check_batch: length mismatch");
    std::vector<uint8_t> ok(results.size());
    if (results.empty()) return {};
    ok_or_throw(vdfgpu_minroot_check_batch(FIELD, results.data(), originals.data(), t.size() == 1 ? nullptr : t.data(),
                                     t.size() == 1 ? t[0] : 0, results.size(), ok.data()),
          "vdfgpu_minroot_check_batch");
    return std::vector<bool>(ok.begin(), ok.end());
  }
  static bool check(const State& result, uint64_t t, const State& original) {
    return check_batch({result}, {t}, {original})[0];
  }
  // inverse_eval (minroot.rs:363-365) for many chains
  static std::vector<State> inverse_eval_batch(const std::vector<State>& results, uint64_t t) {
    std::vector<State> out(results.size());
    if (results.empty()) return out;
    ok_or_throw(vdfgpu_minroot_inverse_eval_batch(FIELD, results.data(), t, results.size(), out.data()),
          "vdfgpu_minroot_inverse_eval_batch");
    return out;
  }
  static State inverse_eval(const State& x, uint64_t t) { return inverse_eval_batch({x}, t)[0]; }
};
using PallasVDF = MinRootVDF<VDFGPU_FQ>;  // modulus of Fq, minroot.rs:38-40
using VestaVDF = MinRootVDF<VDFGPU_FP>;   // modulus of Fp, minroot.rs:199-201

template <class V>
struct Evaluation {  // minroot.rs:376-439 (the slow `eval` stays with the caller: it is sequential host work)
  State result;
  uint64_t t;
  bool verify(const State& original) const { return V::check(result, t, original); }  // :424-426
  std::optional<Evaluation> append(const Evaluation& other) const {                   // :428-438
    if (other.verify(result)) return Evaluation{other.result, t + other.t};
    return std::nullopt;
  }
};

// ---- commitments (nova CommitGens / commit) -------------------------------------------------------------
class Generators {
 public:
  // gens: pasta_curves affine points, fixed for the life of PublicParams (src/nova/proof.rs:232-237)
  Generators(int curve, const std::vector<Affine>& gens, bool table = true) : curve_(curve) {
    ok_or_throw(vdfgpu_gens_create(curve, gens.data(), gens.size(), table ? VDFGPU_GENS_TABLE : 0, 0, &h_), "vdfgpu_gens_create");
  }
  // synthetic known-discrete-log set (k0 + i d) G, generated on the device (tests / benches)
  Generators(int curve, const Fe& k0_le, const Fe& d_le, size_t n, bool table = true) : curve_(curve) {
    ok_or_throw(vdfgpu_gens_progression(curve, k0_le.data(), d_le.data(), n, table ? VDFGPU_GENS_TABLE : 0, 0, &h_),
          "vdfgpu_gens_progression");
  }
  Generators(const Generators&) = delete;
  Generators& operator=(const Generators&) = delete;
  ~Generators() { if (h_) vdfgpu_gens_destroy(h_); }
  size_t len() const { return vdfgpu_gens_len(h_); }
  int curve() const { return curve_; }
  vdfgpu_gens* handle() const { return h_; }
  // commit(v) = vartime_multiscalar_mul(v, gens[..v.len()])
  Point commit(const std::vector<Fe>& scalars) const {
    Point out{};
    ok_or_throw(vdfgpu_msm(h_, scalars.data(), scalars.size(), out.data()), "vdfgpu_msm");
    return out;
  }
  // asynchronous pair for independent commitments: buffers must stay alive (ideally pinned) until wait(slot)
  void commit_submit(const Fe* scalars, size_t n, Point* out, int slot) const {
    ok_or_throw(vdfgpu_msm_submit(h_, scalars, n, out->data(), slot), "vdfgpu_msm_submit");
  }
  static void commit_wait(int slot) { ok_or_throw(vdfgpu_msm_wait(slot), "vdfgpu_msm_wait"); }

 private:
  int curve_;
  vdfgpu_gens* h_ = nullptr;
};

// pasta_msm::pallas / pasta_msm::vesta: points travel with the call
inline Point pasta_msm(int curve, const std::vector<Affine>& points, const std::vector<Fe>& scalars) {
  if (points.size() != scalars.size()) throw std::invalid_argument("pasta_msm: length mismatch");  // wrapper panics
  Point out{};
  if (curve == VDFGPU_PALLAS) mult_pippenger_pallas(out.data(), points.data(), points.size(), scalars.data(), true);
  else mult_pippenger_vesta(out.data(), points.data(), points.size(), scalars.data(), true);
  return out;
}

// ---- R1CS (nova R1CSShape, RelaxedR1CSWitness) ------------------------------------------------------------
struct CooMatrix {  // Vec<(usize, usize, Scalar)>
  std::vector<uint64_t> rows, cols;
  std::vector<Fe> vals;
};

// Verdict of RelaxedR1CSShape::is_sat_relaxed / R1CSShape::is_sat (the report of vdfgpu_r1cs_is_sat_relaxed):
// rows where Az.Bz != u.Cz + E, and each commitment check as 1 = equal, 0 = different, 2 = not checked
struct SatReport {
  uint64_t bad_rows = 0;
  uint64_t first_bad_row = 0;   // num_cons when no row is violated
  uint64_t comm_W = 2, comm_E = 2;
  bool ok() const { return bad_rows == 0 && comm_W != 0 && comm_E != 0; }
};

class R1CSShape {
 public:
  R1CSShape(int field, size_t num_cons, size_t num_vars, size_t num_io, const CooMatrix& A, const CooMatrix& B,
            const CooMatrix& C)
      : field_(field), cons_(num_cons), vars_(num_vars), io_(num_io) {
    for (const CooMatrix* m : {&A, &B, &C})
      if (m->rows.size() != m->vals.size() || m->cols.size() != m->vals.size())
        throw std::invalid_argument("R1CSShape: COO arrays of different lengths");
    ok_or_throw(vdfgpu_r1cs_create(field, num_cons, num_vars, num_io, A.rows.data(), A.cols.data(), A.vals.data(), A.vals.size(),
                             B.rows.data(), B.cols.data(), B.vals.data(), B.vals.size(), C.rows.data(), C.cols.data(),
                             C.vals.data(), C.vals.size(), &h_),
          "vdfgpu_r1cs_create");
  }
  R1CSShape(const R1CSShape&) = delete;
  R1CSShape& operator=(const R1CSShape&) = delete;
  ~R1CSShape() { if (h_) vdfgpu_r1cs_destroy(h_); }
  size_t num_cons() const { return cons_; }
  size_t num_vars() const { return vars_; }
  size_t num_io() const { return io_; }
  int field() const { return field_; }
  vdfgpu_r1cs* handle() const { return h_; }

  struct Products { std::vector<Fe> Az, Bz, Cz; };
  // multiply_vec(z), z = [W | u | X]
  Products multiply_vec(const std::vector<Fe>& z) const {
    if (z.size() != vars_ + 1 + io_) throw std::invalid_argument("multiply_vec: InvalidWitnessLength");
    Products p{std::vector<Fe>(cons_), std::vector<Fe>(cons_), std::vector<Fe>(cons_)};
    ok_or_throw(vdfgpu_multiply_vec(h_, z.data(), p.Az.data(), p.Bz.data(), p.Cz.data()), "vdfgpu_multiply_vec");
    return p;
  }
  // spartan_with_ipa_pc's compute_eval_table_sparse combined with (r_A, r_B, r_C): the inner sum-check's table,
  // out[y] = sum_x eq_rows[x] (r_A A[x,y] + r_B B[x,y] + r_C C[x,y]) over the columns of z
  std::vector<Fe> bind_rows(const std::vector<Fe>& eq_rows, const std::array<Fe, 3>& r_abc) const {
    if (eq_rows.size() != cons_) throw std::invalid_argument("bind_rows: one eq entry per constraint");
    std::vector<Fe> out(vars_ + 1 + io_);
    ok_or_throw(vdfgpu_r1cs_bind_rows(h_, eq_rows.data(), r_abc.data(), out.data()), "vdfgpu_r1cs_bind_rows");
    return out;
  }
  // commit_T(gens, U1, W1, U2, W2) -> (T, comm_T); u2 = 1
  std::pair<std::vector<Fe>, Point> commit_T(const Generators& gens, const std::vector<Fe>& W1, const Fe& u1,
                                             const std::vector<Fe>& X1, const std::vector<Fe>& W2,
                                             const std::vector<Fe>& X2) const {
    // nova-snark returns NovaError::InvalidWitnessLength here; the C ABI takes no lengths, so check before it reads
    if (W1.size() != vars_ || W2.size() != vars_ || X1.size() != io_ || X2.size() != io_)
      throw std::invalid_argument("commit_T: InvalidWitnessLength");
    if (gens.len() < cons_) throw std::invalid_argument("commit_T: fewer generators than constraints");
    std::vector<Fe> T(cons_);
    Point comm{};
    ok_or_throw(vdfgpu_commit_T(h_, gens.handle(), W1.data(), u1.data(), X1.data(), W2.data(), X2.data(), T.data(), comm.data()),
          "vdfgpu_commit_T");
    return {std::move(T), comm};
  }
  // is_sat_relaxed(gens, U, W): Az.Bz = u.Cz + E per row, comm_W = commit(W), comm_E = commit(E).  E empty means
  // E = 0; gens or a commitment nullptr: that commitment is not checked.  Commitments may be un-normalised Jacobian.
  SatReport is_sat_relaxed(const Generators* gens, const std::vector<Fe>& W, const std::vector<Fe>& E, const Fe& u,
                           const std::vector<Fe>& X, const Point* comm_W, const Point* comm_E) const {
    if (W.size() != vars_ || X.size() != io_ || (!E.empty() && E.size() != cons_))
      throw std::invalid_argument("is_sat_relaxed: InvalidWitnessLength");
    return check(gens, W, E.empty() ? nullptr : E.data(), u.data(), X, comm_W, comm_E);
  }
  // is_sat(gens, U, W) of a fresh instance: Az.Bz = Cz (u = 1, E = 0), comm_W = commit(W)
  SatReport is_sat(const Generators* gens, const std::vector<Fe>& W, const std::vector<Fe>& X, const Point* comm_W) const {
    if (W.size() != vars_ || X.size() != io_) throw std::invalid_argument("is_sat: InvalidWitnessLength");
    return check(gens, W, nullptr, nullptr, X, comm_W, nullptr);
  }

 private:
  SatReport check(const Generators* gens, const std::vector<Fe>& W, const Fe* E, const uint8_t* u,
                  const std::vector<Fe>& X, const Point* comm_W, const Point* comm_E) const {
    if (!gens && (comm_W || comm_E)) throw std::invalid_argument("is_sat: checking a commitment needs the generators");
    if (gens && (gens->len() < cons_ || gens->len() < vars_))
      throw std::invalid_argument("is_sat: fewer generators than max(vars, cons)");
    uint64_t rep[4];
    ok_or_throw(vdfgpu_r1cs_is_sat_relaxed(h_, gens ? gens->handle() : nullptr, W.data(), E, u, X.data(),
                                           comm_W ? comm_W->data() : nullptr, comm_E ? comm_E->data() : nullptr, rep),
                "vdfgpu_r1cs_is_sat_relaxed");
    return SatReport{rep[0], rep[1], rep[2], rep[3]};
  }

  int field_;
  size_t cons_, vars_, io_;
  vdfgpu_r1cs* h_ = nullptr;
};

// RelaxedR1CSWitness::fold on host vectors: W1 += r W2, E1 += r T
inline void fold(int field, std::vector<Fe>& W1, const std::vector<Fe>& W2, std::vector<Fe>& E1,
                 const std::vector<Fe>& T, const Fe& r) {
  if (W1.size() != W2.size() || E1.size() != T.size()) throw std::invalid_argument("fold: length mismatch");
  ok_or_throw(vdfgpu_fold(field, W1.data(), W2.data(), W1.size(), E1.data(), T.data(), E1.size(), r.data()), "vdfgpu_fold");
}

// Device-resident running witness: the witness side of NIFS::prove, one call pair per fold step
class RunningWitness {
 public:
  // The shape and the generators must outlive this object (the library refuses to destroy them while it exists).
  RunningWitness(const R1CSShape& s, const Generators& g) : cons_(s.num_cons()), vars_(s.num_vars()), io_(s.num_io()) {
    ok_or_throw(vdfgpu_running_create(s.handle(), g.handle(), &h_), "vdfgpu_running_create");
  }
  RunningWitness(const RunningWitness&) = delete;
  RunningWitness& operator=(const RunningWitness&) = delete;
  ~RunningWitness() { if (h_) vdfgpu_running_destroy(h_); }
  void set(const std::vector<Fe>& W, const std::vector<Fe>& E, const Fe& u, const std::vector<Fe>& X) {
    if (W.size() != vars_ || E.size() != cons_ || X.size() != io_) throw std::invalid_argument("set: InvalidWitnessLength");
    ok_or_throw(vdfgpu_running_set(h_, W.data(), E.data(), u.data(), X.data()), "vdfgpu_running_set");
  }
  struct Commitments { Point comm_W2, comm_T; };
  // commit(W2), T, commit(T): returns what the random oracle absorbs
  Commitments commit(const std::vector<Fe>& W2, const std::vector<Fe>& X2) {
    if (W2.size() != vars_ || X2.size() != io_) throw std::invalid_argument("commit: InvalidWitnessLength");
    Commitments c{};
    ok_or_throw(vdfgpu_running_commit(h_, W2.data(), X2.data(), c.comm_W2.data(), c.comm_T.data()), "vdfgpu_running_commit");
    return c;
  }
  // W += r W2, E += r T, u += r, X += r X2
  void fold(const Fe& r) { ok_or_throw(vdfgpu_running_finish(h_, r.data()), "vdfgpu_running_finish"); }
  void get(std::vector<Fe>& W, std::vector<Fe>& E, Fe& u, std::vector<Fe>& X) const {
    W.resize(vars_);
    E.resize(cons_);
    X.resize(io_);
    ok_or_throw(vdfgpu_running_get(h_, W.data(), E.data(), u.data(), X.data()), "vdfgpu_running_get");
  }
  // is_sat_relaxed of the resident running instance (nothing is copied back); a commitment nullptr is not checked
  SatReport check(const Point* comm_W, const Point* comm_E) const {
    uint64_t rep[4];
    ok_or_throw(vdfgpu_running_check(h_, comm_W ? comm_W->data() : nullptr, comm_E ? comm_E->data() : nullptr, rep),
                "vdfgpu_running_check");
    return SatReport{rep[0], rep[1], rep[2], rep[3]};
  }

 private:
  size_t cons_, vars_, io_;
  vdfgpu_running* h_ = nullptr;
};

}  // namespace vdf_host
