/* vdfgpu.h -- C ABI of libvdfgpu.so: the B200 (sm_100a) data-parallel hot path of protocol/vdf's Nova
 * prover for the MinRoot VDF.  Plain pointers and sizes only; every entry point names the reference
 * interface it replaces.  The reference is pure Rust (src/minroot.rs, src/nova/proof.rs) and reaches the
 * arithmetic below through nova-snark 0.8 / pasta-msm 0.1 / pasta_curves 0.4 (Cargo.toml:15,17,18); the
 * Rust-side bindings a maintainer would add are shown in INTEGRATION.md.
 *
 * Data layouts (pasta_curves with feature "repr-c", Cargo.toml:17):
 *   field element  32 B   four little-endian u64 limbs, Montgomery form (value * 2^256 mod m)
 *   affine point   72 B   { x: 32 B, y: 32 B, infinity: u8, 7 B padding }
 *   point          96 B   Jacobian { X, Y, Z }, identity <=> Z == 0.  Results are written normalised:
 *                         (x, y, 1) or (0, 0, 0), so equal group elements have equal bytes.
 *   State<F>       96 B   { x, y, i } (src/minroot.rs:267-272)
 *
 * Curves: VDFGPU_PALLAS (coordinates in Fp, scalars in Fq), VDFGPU_VESTA (coordinates in Fq, scalars in
 * Fp).  Fields: VDFGPU_FP (Pallas base), VDFGPU_FQ (Pallas scalar; the field of PallasVDF,
 * src/minroot.rs:38).
 *
 * Errors: every int-returning function returns 0 on success and a negative code on failure;
 * vdfgpu_last_error() returns a thread-local message.  There is NO CPU fallback: without a usable CUDA
 * device every compute call fails with VDFGPU_ERR_CUDA.
 *
 * Memory: "host" pointers are ordinary host memory owned by the caller for the duration of the call
 * (pinned memory makes the copies faster); "_dev" entry points take device pointers and enqueue on the
 * calling thread's stream (vdfgpu_set_stream) without synchronising.  Handles are owned by the library and
 * freed by the matching *_destroy.  Calls on one thread are ordered; the library keeps no pointer after return
 * (except vdfgpu_msm_submit, whose buffers it owns until vdfgpu_msm_wait of that slot).
 *
 * Threads and devices: ONE GPU per process (vdfgpu_init(device); a call before vdfgpu_init binds device 0, which
 * is what the literal pasta-msm entry points need).  Every entry point may be called from any thread: the library
 * takes an internal lock only while it ENQUEUES work and waits for the GPU after releasing it, so calls from
 * several threads overlap on the device; the stream is a per-THREAD setting; the caller's current CUDA device is
 * restored before a call returns.  Ordering: the work a call does on a handle's own device state (a running instance's
 * W, E, u, X, W2, T) is ordered behind the previous call on that handle whatever the stream or thread of either, so
 * vdfgpu_running_finish may return before its fold has run and the next call may come from another stream or thread.
 * Device buffers the caller passes to "_dev" entry points are ordered by the caller's stream only: whatever writes
 * them on another stream must be made visible to it (an event) before the call.  A handle must not be destroyed while another thread uses it; a generator set or
 * shape held by a running instance (or a set in use by vdfgpu_ipa_prove[_dev]) cannot be destroyed (VDFGPU_ERR_STATE)
 * until that instance is (that call has returned).
 *
 * Inputs: every 32-byte field element must be the canonical Montgomery image of a value < m, as pasta_curves'
 * from_repr guarantees on the Rust side.  The MinRoot verdict entry points check this themselves (a non-canonical
 * State gives ok = 0), and so does vdfgpu_ipa_verify_batch for its proofs; the other entry points do not.
 *
 * Limits: point references are 31 bits, so windows * points of one generator set must stay below 2^31 (a table
 * set of 2^26 points x 13 levels uses 41 %); shard larger sets by point range (vdfgpu_msm_range_dev / one set per
 * GPU) and add the partial results with vdfgpu_point_sum.
 */
#ifndef VDFGPU_H
#define VDFGPU_H

#include <stdbool.h>
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VDFGPU_PALLAS 0
#define VDFGPU_VESTA 1
#define VDFGPU_FP 0
#define VDFGPU_FQ 1

#define VDFGPU_OK 0
#define VDFGPU_ERR_ARG (-1)
#define VDFGPU_ERR_CUDA (-2)
#define VDFGPU_ERR_STATE (-3)

/* generator-set flags */
#define VDFGPU_GENS_TABLE 1u /* precompute 2^(c*w) * P_i levels (W x memory, one shared bucket set) */
#define VDFGPU_GENS_RAW_JACOBIAN 2u /* results as un-normalised Jacobian (X, Y, Z), like pasta-msm returns them: skips
                                     * the single-thread field inversion (~0.13 ms); the caller's to_affine() normalises */

typedef struct vdfgpu_gens vdfgpu_gens;   /* device-resident commitment generators (nova CommitGens) */
typedef struct vdfgpu_r1cs vdfgpu_r1cs;   /* device-resident R1CS shape in CSR (nova R1CSShape) */
typedef struct vdfgpu_running vdfgpu_running;   /* device-resident running witness (nova RelaxedR1CSWitness) */

/* ---- context -------------------------------------------------------------------------------------- */
int vdfgpu_init(int device);              /* bind this process to one GPU (one process per GPU) */
int vdfgpu_shutdown(void);
int vdfgpu_device_count(void);
const char* vdfgpu_last_error(void);
const char* vdfgpu_version(void);
int vdfgpu_set_stream(void* cuda_stream); /* cudaStream_t for the CALLING THREAD's subsequent work; NULL = library stream */
int vdfgpu_synchronize(void);             /* waits for the calling thread's stream */
/* frees the preallocated MSM workspaces (one per stream that ran an MSM) and the cached pool memory */
int vdfgpu_trim(void);
uint64_t vdfgpu_launch_count(void);       /* kernels launched by this library so far */

/* ---- a4: MSM.  Replaces pasta-msm's extern "C" mult_pippenger_{pallas,vesta}, the backend of nova's
 * Group::vartime_multiscalar_mul used by commit(W) / commit(T) (reached from src/nova/proof.rs:342-349).
 * Same symbol names and signature as pasta-msm 0.1.1 so its Rust wrapper links against this object. ---- */
void mult_pippenger_pallas(void* out_point96, const void* points_affine72, size_t npoints,
                           const void* scalars32, bool is_mont);
void mult_pippenger_vesta(void* out_point96, const void* points_affine72, size_t npoints,
                          const void* scalars32, bool is_mont);

/* The literal entry points keep the generator sets they have seen resident (nova passes the same Vec every time):
 * see "drop-in cache" in vdf_b200/csrc/api_core.cu.  Environment: VDFGPU_DROPIN_CACHE=0 (off),
 * VDFGPU_DROPIN_VERIFY=sample|full|off (how a cached set is re-validated against the caller's memory; default
 * sample), VDFGPU_DROPIN_ENTRIES (LRU size, default 4). */
int vdfgpu_dropin_cache_clear(void);
int vdfgpu_dropin_cache_stats(uint64_t* hits, uint64_t* misses, uint64_t* entries);

/* Generators are fixed for the life of PublicParams (src/nova/proof.rs:232-237): upload/repack once.
 * window_bits (2..24, 0 = by size) applies to VDFGPU_GENS_TABLE sets, whose table levels are built for it.  A plain set
 * ignores it and picks the window size per call from the number of scalars; vdfgpu_gens_window_bits reports either. */
int vdfgpu_gens_create(int curve, const void* points_affine72_host, size_t n, uint32_t flags,
                       uint32_t window_bits /* 0 = auto */, vdfgpu_gens** out);
/* synthetic set P_i = (k0 + i*d) * G, G = (-1, 2), generated on the device (bench/tests, SURVEY 8d C2);
 * k0 and d are 32-byte little-endian canonical (non-Montgomery) integers */
int vdfgpu_gens_progression(int curve, const void* k0_le32, const void* d_le32, size_t n, uint32_t flags,
                            uint32_t window_bits, vdfgpu_gens** out);
int vdfgpu_gens_export(const vdfgpu_gens* g, size_t first, size_t count, void* points_affine72_host);
size_t vdfgpu_gens_len(const vdfgpu_gens* g);
uint32_t vdfgpu_gens_window_bits(const vdfgpu_gens* g, size_t n);
/* batched-affine halving rounds an n-scalar commitment over g runs before its XYZZ accumulation (measurement) */
uint32_t vdfgpu_gens_affine_rounds(const vdfgpu_gens* g, size_t n);
int vdfgpu_gens_destroy(vdfgpu_gens* g);

/* commit(v) = sum_i v_i * gens[i] over the first n generators; scalars in Montgomery form */
int vdfgpu_msm(vdfgpu_gens* g, const void* scalars32_host, size_t n, void* out_point96_host);
int vdfgpu_msm_dev(vdfgpu_gens* g, const void* scalars32_dev, size_t n, void* out_point96_dev);
/* Asynchronous form of vdfgpu_msm for callers with several independent commitments: submit returns once the
 * work is enqueued (use pinned host memory), wait blocks until out_point96_host of that slot is written.  Every
 * slot has its own stream: the upload AND the latency-bound stages of slot k+1 overlap the kernels of slot k.
 * slot in [0, 4); a busy slot must be waited before reuse; host buffers of a slot stay owned by the library until
 * its wait returns. */
int vdfgpu_msm_submit(vdfgpu_gens* g, const void* scalars32_host, size_t n, void* out_point96_host, int slot);
int vdfgpu_msm_wait(int slot);
/* k <= 4 scalar vectors (lengths lens[j]) over the same generators in ONE pass: k commitments for the latency
 * of one MSM.  nova commits to W and T of one NIFS::prove with the same generators. */
int vdfgpu_msm_batch_dev(vdfgpu_gens* g, const void* const* scalars32_dev, const size_t* lens, uint32_t k,
                         void* out_points96_dev);
/* point range [first, first+n) of the set: the shard a rank owns in the multi-GPU MSM (SURVEY 8e) */
int vdfgpu_msm_range_dev(vdfgpu_gens* g, size_t first, const void* scalars32_dev, size_t n,
                         void* out_point96_dev);
/* (X, Y, Z) -> (X / Z^2, Y / Z^3, 1) in place on `count` HOST points, computed on the host (no GPU needed): what the
 * host entry points apply to their results after the copy has landed -- a field inversion is one sequential chain of
 * ~335 multiplications, 0.12 ms in one GPU thread against ~15 us on a CPU core -- and what a caller applies to the
 * un-normalised results of a VDFGPU_GENS_RAW_JACOBIAN set or of the _dev entry points when it wants canonical bytes.
 * VDFGPU_HOST_NORMALISE=0 moves the normalisation of the host entry points back onto the device. */
int vdfgpu_point_normalise_host(int curve, void* points96_host, size_t count);
/* out = sum of k points (combining per-GPU partial results; also instance-side additions) */
int vdfgpu_point_sum(int curve, const void* points96_host, size_t k, void* out_point96_host);

/* ---- a5-a7: R1CS.  Replaces nova-snark R1CSShape::{multiply_vec, commit_T} and
 * RelaxedR1CSWitness::fold (reached from src/nova/proof.rs:342-349).  COO triples as nova stores them
 * (row: usize, col: usize, val: Scalar); column j < vars is W[j], j == vars is u, j > vars is X. ---- */
int vdfgpu_r1cs_create(int field, size_t num_cons, size_t num_vars, size_t num_io,
                       const uint64_t* a_rows, const uint64_t* a_cols, const void* a_vals32, size_t a_nnz,
                       const uint64_t* b_rows, const uint64_t* b_cols, const void* b_vals32, size_t b_nnz,
                       const uint64_t* c_rows, const uint64_t* c_cols, const void* c_vals32, size_t c_nnz,
                       vdfgpu_r1cs** out);
int vdfgpu_r1cs_destroy(vdfgpu_r1cs* s);
/* (Az, Bz, Cz) for z = [W | u | X] given as one host vector of vars+1+io elements */
int vdfgpu_multiply_vec(const vdfgpu_r1cs* s, const void* z_host, void* Az_host, void* Bz_host,
                        void* Cz_host);
/* T = Az1.Bz2 + Az2.Bz1 - u1.Cz2 - u2.Cz1 (u2 = 1) and comm_T = MSM(T, gens); gens may be NULL to skip
 * the commitment.  T_host may be NULL. */
int vdfgpu_commit_T(const vdfgpu_r1cs* s, vdfgpu_gens* gens, const void* W1_host, const void* u1_host,
                    const void* X1_host, const void* W2_host, const void* X2_host, void* T_host,
                    void* comm_T_point96_host);
/* W1 <- W1 + r*W2 (nW elements), E1 <- E1 + r*T (nE elements), in place on host buffers */
int vdfgpu_fold(int field, void* W1_host, const void* W2_host, size_t nW, void* E1_host,
                const void* T_host, size_t nE, const void* r32_host);

/* device-pointer variants (no copies, no synchronisation): what a device-resident prover and bench.py's
 * HBM-roofline leg call.  uX = [u | X] (1 + io elements), uX2 = [1 | X2]. */
int vdfgpu_multiply_vec_dev(const vdfgpu_r1cs* s, const void* W_dev, const void* uX_dev, void* AzBzCz_dev);

/* Spartan's inner sum-check table (SURVEY 8f rank 2; nova-snark 0.8 spartan_with_ipa_pc: compute_eval_table_sparse
 * combined with r_A, r_B, r_C [R], reached from CompressedSNARK::prove, /root/reference/src/nova/proof.rs:363):
 *   out[y] = sum_x eq_rows[x] * (r_abc[0] A[x,y] + r_abc[1] B[x,y] + r_abc[2] C[x,y]),  y < vars + 1 + io.
 * eq_rows: cons elements (the eq table of the outer challenge, vdfgpu_eq_evals), r_abc: 3 elements, out: vars+1+io
 * elements, all 32-byte Montgomery.  The _dev form works on device pointers on the calling thread's stream and needs
 * a scratch vector of 3 * cons elements. */
int vdfgpu_r1cs_bind_rows(const vdfgpu_r1cs* s, const void* eq_rows_host, const void* r_abc_host, void* out_host);
int vdfgpu_r1cs_bind_rows_dev(const vdfgpu_r1cs* s, const void* eq_rows_dev, const void* r_abc_dev, void* scratch_dev,
                              void* out_dev);
int vdfgpu_cross_term_dev(const vdfgpu_r1cs* s, const void* W1_dev, const void* uX1_dev, const void* W2_dev,
                          const void* uX2_dev, void* T_dev);
int vdfgpu_fold_dev(int field, void* W1_dev, const void* W2_dev, size_t nW, void* E1_dev, const void* T_dev,
                    size_t nE, const void* r32_dev);

/* Device-resident running instance for a chain of fold steps: W and E never leave HBM between steps.
 * One step = what NIFS::prove does with the witness: commit_T against a fresh (W2, X2), then fold with
 * the verifier challenge r (computed by the host random oracle from comm_T, so it arrives later). */
int vdfgpu_running_create(const vdfgpu_r1cs* s, vdfgpu_gens* gens, vdfgpu_running** out);
int vdfgpu_running_destroy(vdfgpu_running* f);
int vdfgpu_running_set(vdfgpu_running* f, const void* W_host, const void* E_host, const void* u_host,
                            const void* X_host);
int vdfgpu_running_get(const vdfgpu_running* f, void* W_host, void* E_host, void* u_host, void* X_host);
/* CompressedSNARK::prove of the running instance without reading it back: vdfgpu_running_spartan_prove, after the
 * sum-check and IPA callback types below */
/* upload fresh witness, commit to it, compute T and comm_T; W2/T stay on the device for running_finish */
int vdfgpu_running_commit(vdfgpu_running* f, const void* W2_host, const void* X2_host,
                       void* comm_W2_point96_host, void* comm_T_point96_host);
/* W <- W + r*W2, E <- E + r*T, u <- u + r, X <- X + r*X2; returns once enqueued (the next call on f, on any stream or
 * thread, is ordered behind it) */
int vdfgpu_running_finish(vdfgpu_running* f, const void* r32_host);

/* ---- RecursiveSNARK::verify (src/nova/proof.rs:382): RelaxedR1CSShape::is_sat_relaxed / R1CSShape::is_sat [R] of
 * the primary and secondary running instances and of the last fresh secondary instance.  Each check fills a report of
 * four uint64_t:
 *   [0] rows with Az.Bz != u.Cz + E      [1] smallest such row, num_cons when there is none
 *   [2] comm_W == commit(W): 1 yes, 0 no, 2 not checked       [3] comm_E == commit(E): same coding
 * An unsatisfied instance is a verdict, not an error: the call returns 0.
 * E_host NULL => E = 0; u_host NULL => u = 1 (both NULL: the strict R1CS check of a fresh instance).
 * gens NULL => no commitment check (comm pointers must be NULL); comm_E96_host requires E_host; gens must hold at least
 * max(num_vars, num_cons) points of the curve whose scalar field is the shape's.
 * Commitments are compared as group elements: the caller's points may be un-normalised Jacobian. ---- */
int vdfgpu_r1cs_is_sat_relaxed(const vdfgpu_r1cs* s, vdfgpu_gens* gens, const void* W_host, const void* E_host,
                               const void* u_host, const void* X_host, const void* comm_W96_host,
                               const void* comm_E96_host, uint64_t* report4_host);
/* row check only, on the calling thread's stream, no synchronisation; the call initialises counts2_dev
 * ([0] violating rows, [1] smallest violating row); E_dev may be NULL (E = 0); uX = [u | X] */
int vdfgpu_r1cs_is_sat_relaxed_dev(const vdfgpu_r1cs* s, const void* W_dev, const void* E_dev, const void* uX_dev,
                                   uint64_t* counts2_dev);
/* the same check on a device-resident running instance (W, E, u, X never leave HBM) with its generators; either
 * commitment may be NULL (not checked).  Before vdfgpu_running_set: VDFGPU_ERR_STATE. */
int vdfgpu_running_check(const vdfgpu_running* f, const void* comm_W96_host, const void* comm_E96_host,
                         uint64_t* report4_host);

/* SURVEY 8f rank 1 -- the step-circuit part of the fresh witness never crosses PCIe.  A bank holds, for all n steps
 * of one proof, the 4t+1 values InverseMinRootCircuit::synthesize allocates (src/nova/proof.rs:107-126, :162-189),
 * generated on the device from the steps' input states (x, y, i) -- the circuits of a proof are independent once the
 * VDF states are known (src/nova/proof.rs:284-296).  Creation is asynchronous (own stream).
 * vdfgpu_running_commit_step is vdfgpu_running_commit with
 *   W2 = [ W2_host[0, step_offset) | bank[step] | W2_host[step_offset + 4t + 1, vars) ]
 * W2_host has the full length; its step range is neither read nor transferred. */
typedef struct vdfgpu_witness_bank vdfgpu_witness_bank;
int vdfgpu_witness_bank_create(int field, const void* z_in_state96_host, uint64_t t, size_t n,
                               vdfgpu_witness_bank** out);
int vdfgpu_witness_bank_destroy(vdfgpu_witness_bank* b);
int vdfgpu_witness_bank_read(const vdfgpu_witness_bank* b, size_t first_step, size_t count, void* out_fe32_host);
int vdfgpu_running_commit_step(vdfgpu_running* f, const vdfgpu_witness_bank* bank, size_t step, size_t step_offset,
                               const void* W2_host, const void* X2_host, void* comm_W2_point96_host,
                               void* comm_T_point96_host);

/* ---- SURVEY 8f rank 2: sum-check building blocks of CompressedSNARK::prove (src/nova/proof.rs:360-368 -> nova-snark 0.8
 * spartan_with_ipa_pc; that crate is not under the reference tree: semantics restated in vdf_b200/csrc/sumcheck.cuh).
 * Tables are multilinear polynomials in evaluation form, 2^ell field elements, most significant variable first.
 *   eq_evals        out[idx] = prod_j (bit_j(idx) ? r_j : 1 - r_j)                      (EqPolynomial::evals)
 *   sumcheck_cubic  ell rounds of prove_cubic_with_additive_term with comb(A,B,C,D) = A (B C - D): every round the
 *                   library computes (e0, e2, e3), hands them to round_fn -- which owns the transcript: it forms the
 *                   round polynomial from [e0, claim - e0, e2, e3], absorbs it, squeezes the challenge and writes it to
 *                   r_out_fe32 (return 0; non-zero aborts with VDFGPU_ERR_STATE) -- and binds the top variable of all
 *                   four tables to it.  final_evals receives A[0], B[0], C[0], D[0].  The tables are consumed.
 *   sumcheck_quad   the same with comb(A,B) = A B and evaluations (e0, e2)               (prove_quad)
 *   poly_evaluate   <eq(r), P>                                                          (MultilinearPolynomial::evaluate)
 * round_fn runs on the calling thread, outside the library's lock. */
typedef int (*vdfgpu_round_fn)(void* user, size_t round, const void* evals_fe32, size_t n_evals, void* r_out_fe32);
int vdfgpu_eq_evals(int field, const void* r_host, size_t ell, void* out_host);
int vdfgpu_eq_evals_dev(int field, const void* r_host, size_t ell, void* out_dev);
int vdfgpu_sumcheck_cubic(int field, const void* A_host, const void* B_host, const void* C_host, const void* D_host,
                          size_t ell, vdfgpu_round_fn round_fn, void* user, void* final_evals4_host);
int vdfgpu_sumcheck_cubic_dev(int field, void* A_dev, void* B_dev, void* C_dev, void* D_dev, size_t ell,
                              vdfgpu_round_fn round_fn, void* user, void* final_evals4_host);
int vdfgpu_sumcheck_quad(int field, const void* A_host, const void* B_host, size_t ell, vdfgpu_round_fn round_fn,
                         void* user, void* final_evals2_host);
int vdfgpu_sumcheck_quad_dev(int field, void* A_dev, void* B_dev, size_t ell, vdfgpu_round_fn round_fn, void* user,
                             void* final_evals2_host);
int vdfgpu_poly_evaluate(int field, const void* poly_host, const void* r_host, size_t ell, void* out_host);
int vdfgpu_poly_evaluate_dev(int field, const void* poly_dev, const void* r_host, size_t ell, void* out_host);
/* One round of the inner-product argument behind spartan_with_ipa_pc's polynomial-commitment opening halves vectors
 * and generators with the challenge r:  a' = r a_L + r^-1 a_R (vec_lincomb: out[i] = x a[i] + y b[i]),
 * c = <a_L, b_R> (inner_product), G'_i = r^-1 G_L,i + r G_R,i (points_lincomb: out[i] = w1 P[i] + w2 Q[i], affine in,
 * affine out -- CommitGens::fold, which nova computes as n/2 two-point vartime_multiscalar_muls).  The two MSMs of a
 * round (L and R) go through vdfgpu_msm / mult_pippenger_*. */
int vdfgpu_vec_lincomb(int field, const void* a_host, const void* b_host, size_t n, const void* x32_host,
                       const void* y32_host, void* out_host);
int vdfgpu_inner_product(int field, const void* a_host, const void* b_host, size_t n, void* out32_host);
int vdfgpu_points_lincomb(int curve, const void* P_affine72_host, const void* Q_affine72_host, size_t n,
                          const void* w1_32_host, const void* w2_32_host, void* out_affine72_host);
/* The whole inner-product argument (spartan_with_ipa_pc's polynomial-evaluation argument [R]) on a resident set g:
 * n = 2^ell; a, b: n elements of the scalar field of g's curve (Montgomery); g holds at least n + 1 points, G_k is
 * point k and U0 = G_n is nova's gens_c; U = u_scale U0 (nova scales gens_c by a transcript scalar before the rounds;
 * a caller without that step passes u_scale = 1).  Round j = 0 .. ell-1, m = n / 2^j, h = m / 2:
 *   c_L = <a[0,h), b[h,m)>, c_R = <a[h,m), b[0,h)>
 *   L = <a[0,h), G'[h,m)> + c_L U,  R = <a[h,m), G'[0,h)> + c_R U
 *   round_fn(user, j, L, R, r_out) -- the caller's transcript: absorbs L and R, writes the challenge r != 0
 *   a <- r a_L + r^-1 a_R,  b <- r^-1 b_L + r b_R,  G' <- r^-1 G'_L + r G'_R
 * a_hat = a[0] after ell rounds.  L and R are normalised as vdfgpu_msm returns them (identity = 96 zero bytes), for
 * every set layout including VDFGPU_GENS_RAW_JACOBIAN.  round_fn runs on the calling thread, outside the library's
 * lock; a non-zero return, r = 0 or a non-canonical r (>= the group order) ends the call with VDFGPU_ERR_STATE.  g
 * stays referenced for the whole call: vdfgpu_gens_destroy from another thread meanwhile returns VDFGPU_ERR_STATE.  ell = 0: a_hat = a[0], round_fn is not called
 * (and may be NULL).  The _dev form works on device vectors on the calling thread's stream and consumes them; the host
 * form takes ell <= 30.
 * ipa_gens_hat: the verifier's folded generator G_hat = <s, G[0,n)> from the ell challenges (g holds at least n
 * points), s_k = prod_j (bit_j(k) ? r_j : r_j^-1) with bit_0 the most significant of the ell bits (nova's s); a
 * challenge that is 0 or non-canonical is VDFGPU_ERR_ARG. */
typedef int (*vdfgpu_ipa_round_fn)(void* user, size_t round, const void* L_point96, const void* R_point96,
                                   void* r_out32);
int vdfgpu_ipa_prove(vdfgpu_gens* g, const void* a_host, const void* b_host, size_t ell, const void* u_scale32_host,
                     vdfgpu_ipa_round_fn round_fn, void* user, void* a_hat32_host);
int vdfgpu_ipa_prove_dev(vdfgpu_gens* g, void* a_dev, void* b_dev, size_t ell, const void* u_scale32_host,
                         vdfgpu_ipa_round_fn round_fn, void* user, void* a_hat32_host);
int vdfgpu_ipa_gens_hat(vdfgpu_gens* g, const void* r_host, size_t ell, void* out_point96_host);
/* ipa_verify_batch: verifies k inner-product arguments over the same set g (at least 2^ell + 1 points, U0 = G_n) in
 * one call.  Proof q: comm_a[q] (the commitment to a), L[q][j] and R[q][j] (j < ell, proof-major), a_hat[q]; its
 * instance: c[q] = <a, b>, b_hat[q] = <b, s_q>, u_scale[q] (U = u_scale U0); r[q][j]: the challenges the caller's
 * transcript derived from L and R.  Proof q is valid iff
 *   a_hat G_hat + u_scale (a_hat b_hat - c) U0 - comm_a - sum_j (r_j^2 L_j + r_j^-2 R_j) = O,   G_hat = <s_q, G[0,n)>
 * (nova's InnerProductArgument::verify with P = comm_a + c U), s_q as for ipa_gens_hat.  b_hat is an input because b
 * is the caller's: for b = eq(x), b_hat = prod_j ((1 - x_j) r_j^-1 + x_j r_j); for b = sum_i rho_i eq(x_i) (two
 * evaluation claims folded into one) the sum of those terms; a table shorter than 2^ell, zero-padded at the top, is
 * eq over x with leading zero coordinates.  Points are 96-byte Jacobian (X, Y, Z), normalised or not; the identity is
 * Z = 0 (96 zero bytes, as vdfgpu_msm returns it).  Scalars are 32-byte Montgomery in g's scalar field.
 * The k equations are checked as ONE weighted sum, sum_q w_q (equation q) = O: one MSM over G[0, n] and one over the
 * k (2 ell + 1) caller points.  If that sum is not O, each proof is checked alone (MSMs in batches of four: about k/4
 * extra MSM passes over the set, paid only by a failing batch).  ok_out[q] = 1 iff proof q is valid; the verdicts
 * fail closed: whenever the call returns an error, every ok_out[q] it could write is 0.
 * Verdicts and errors: a malformed proof is a verdict, not an error -- a point with a coordinate >= p or off
 * y^2 = x^3 + 5, or a non-canonical a_hat, c, b_hat or u_scale gives ok_out[q] = 0 for that proof only and leaves it
 * out of the weighted sum.  VDFGPU_ERR_ARG, before any device work: a null pointer, k = 0, ell > 40, fewer than
 * 2^ell + 1 points in g, a challenge that is 0 or >= the group order, a weight that is 0 or >= the group order.
 * Soundness: the weights must be uniform and unpredictable to whoever produced the proofs (the OS CSPRNG, e.g.
 * OsRng); a batch that contains an invalid proof then passes with probability at most 1 / order.  Weights the prover
 * can predict let two invalid proofs cancel.  The library never generates weights.  g stays referenced for the call,
 * which runs on the calling thread's stream. */
int vdfgpu_ipa_verify_batch(vdfgpu_gens* g, size_t ell, size_t k, const void* comm_a96_host, const void* L96_host,
                            const void* R96_host, const void* r32_host, const void* a_hat32_host, const void* c32_host,
                            const void* b_hat32_host, const void* u_scale32_host, const void* w32_host,
                            uint8_t* ok_out_host);

/* RelaxedR1CSSNARK::prove of the running instance (CompressedSNARK::prove, src/nova/proof.rs:363 -> nova-snark 0.8
 * spartan_with_ipa_pc [R]; the math is restated in vdf_b200/csrc/sumcheck.cuh) in ONE call, the transcript left to the
 * caller's callbacks.  Padded layout (nova's R1CSShape::pad [R]): m = the next power of two >= max(num_vars, num_cons);
 * column c of the shape is column c if c < num_vars, else c + (m - num_vars), so z = [W | 0 | u | X | 0] has 2m entries;
 * ell_x = log2 m, ell_y = ell_x + 1; 1 + num_io <= m is required.  In order:
 *   1. snapshot: W and E (zero-padded to m) and u, X are copied on the device behind the instance's previous call; the
 *      proof reads only the snapshot (a later running_commit / running_finish cannot change it).
 *   2. outer sum-check of sum_x eq(tau, x) (Az Bz - (u Cz + E))(x) = 0, ell_x rounds: sc_round(user, j, (e0, e2, e3),
 *      3, r_out) -> r_x.  claim_Az, claim_Bz: the bound tables; claim_Cz = Cz(r_x), eval_E = E(r_x).
 *      claims(user, VDFGPU_SPARTAN_OUTER, (claim_Az, claim_Bz, claim_Cz, eval_E), 4, (r_A, r_B, r_C), 3).
 *   3. inner sum-check of sum_y M(y) z(y) with M(y) = sum_x eq(r_x, x) (r_A A + r_B B + r_C C)[x, y], ell_y rounds:
 *      sc_round(user, j, (e0, e2), 2, r_out) -> r_y (round indices restart at 0).  r_y' = r_y[1..].
 *   4. eval_W = W(r_y'), T = <E, eq(r_y')> + <W, eq(r_x)>: claims(user, VDFGPU_SPARTAN_EVAL, (eval_W, T), 2, rho, 1).
 *   5. the two claims E(r_x) = eval_E, W(r_y') = eval_W folded into one (nova's fold of two inner-product instances
 *      [R]): a = E + rho W, b = eq(r_x) + rho eq(r_y'), c = eval_E + rho T + rho^2 eval_W; the caller forms
 *      comm_a = comm_E + rho comm_W.  claims(user, VDFGPU_SPARTAN_IPA, c, 1, u_scale, 1).
 *   6. vdfgpu_ipa_prove of (a, b) over ipa_gens with u_scale: ipa_round as there; a_hat into a_hat32_host.
 * All values are 32-byte Montgomery elements of the shape's field.  ipa_gens: the curve whose scalar field is the
 * shape's, at least m + 1 points (U0 = G_m); its first m points must be the instance's commitment generators (it may be
 * the instance's own set when that holds m + 1 points).  tau: ell_x elements.  Callbacks run on the calling thread,
 * outside the library's lock; a non-zero return, a non-canonical value returned, or an IPA challenge of 0 ends the call
 * with VDFGPU_ERR_STATE.  VDFGPU_ERR_ARG before any device work: a null pointer, ipa_gens of the wrong curve or with
 * fewer than m + 1 points, 1 + num_io > m.  Before vdfgpu_running_set: VDFGPU_ERR_STATE.  The shape, ipa_gens and f
 * stay referenced for the whole call: destroying any of them meanwhile returns VDFGPU_ERR_STATE.  The instance itself
 * is left unchanged. */
typedef int (*vdfgpu_spartan_claims_fn)(void* user, int stage, const void* in_fe32, size_t n_in, void* out_fe32,
                                        size_t n_out);
enum { VDFGPU_SPARTAN_OUTER = 0, VDFGPU_SPARTAN_EVAL = 1, VDFGPU_SPARTAN_IPA = 2 };
int vdfgpu_running_spartan_prove(vdfgpu_running* f, vdfgpu_gens* ipa_gens, const void* tau_host,
                                 vdfgpu_round_fn sc_round, vdfgpu_spartan_claims_fn claims,
                                 vdfgpu_ipa_round_fn ipa_round, void* user, void* a_hat32_host);
/* The sparse part of RelaxedR1CSSNARK::verify [R]: out = (A(r_x, r_y), B(r_x, r_y), C(r_x, r_y)) over the padded layout
 * above, A(r_x, r_y) = sum over entries (x, c, v) of v eq(r_x, x) eq(r_y, col(c)); r_x: ell_x elements, r_y: ell_x + 1
 * (most significant variable first).  1 + num_io > m: VDFGPU_ERR_ARG. */
int vdfgpu_r1cs_evaluate(const vdfgpu_r1cs* s, const void* rx_host, const void* ry_host, void* out3_host);
/* The same for k points in one pass: out[q] = (A, B, C)(r_x[q], r_y[q]), q < k; rx: [k][ell_x], ry: [k][ell_x + 1],
 * out: [k][3], proof-major.  eq(r_x[q]) and eq(r_y[q]) are never written out: each is read from two half tables of
 * about 2^(ell / 2) entries.  k = 0 or 1 + num_io > m: VDFGPU_ERR_ARG. */
int vdfgpu_r1cs_evaluate_batch(const vdfgpu_r1cs* s, size_t k, const void* rx_host, const void* ry_host,
                               void* out3_host);

/* RelaxedR1CSSNARK::verify [R] of k proofs over one shape in one call, the transcript left to the caller: it replays
 * each proof through its own transcript and hands the library the challenges it squeezed.  Notation and padded layout
 * as for vdfgpu_running_spartan_prove (ell_x = log2 m, derived from the shape; ell_y = ell_x + 1; r_y' = r_y[1..]).
 * Records are proof-major; scalars are 32-byte Montgomery elements of the shape's field, points 96-byte Jacobian
 * (X, Y, Z) of ipa_gens' curve, normalised or not, the identity Z = 0.
 *   inst:   [k][1 + num_io]  u, X
 *   points: [k][POINTS]      comm_W, comm_E, L_0 .. L_{ell_x - 1}, R_0 .. R_{ell_x - 1}
 *   proof:  [k][PROOF_FES]   outer rounds (e0, e2, e3) x ell_x, claim_Az, claim_Bz, claim_Cz, eval_E, inner rounds
 *                            (e0, e2) x ell_y, eval_W, T, a_hat -- what vdfgpu_running_spartan_prove hands to its
 *                            callbacks, in that order (c is not part of it: the library derives it)
 *   chal:   [k][CHAL_FES]    tau x ell_x, r_x x ell_x, r_A, r_B, r_C, r_y x ell_y, rho, u_scale, the IPA's r_j x ell_x
 *   w:      [k]              batch weights
 * Proof q is valid iff
 *   1. outer sum-check: starting from claim 0, each round's e1 = claim - e0 and the next claim is the degree-3
 *      interpolant through e0, e1, e2, e3 at r_x[j]; the final claim = eq(tau, r_x) (claim_Az claim_Bz - u claim_Cz -
 *      eval_E);
 *   2. inner sum-check: the same (degree 2) from r_A claim_Az + r_B claim_Bz + r_C claim_Cz at r_y;
 *   3. its final claim = (r_A A + r_B B + r_C C)(r_x, r_y) z(r_y), z(r_y) = (1 - r_y[0]) eval_W + r_y[0] eval_X,
 *      eval_X = the zero-padded (u, X) at r_y' (A, B, C as vdfgpu_r1cs_evaluate, for all proofs in one pass);
 *   4. the opening is valid (the equation of vdfgpu_ipa_verify_batch over ipa_gens, ell = ell_x) with comm_a = comm_E +
 *      rho comm_W, c = eval_E + rho T + rho^2 eval_W, b_hat = prod_j ((1 - r_x,j) r_j^-1 + r_x,j r_j) + rho prod_j
 *      ((1 - r_y',j) r_j^-1 + r_y',j r_j), and u_scale; c and b_hat are derived by the library, never taken from the
 *      caller.
 * Checks 1, 2 and the derivations run on the host, O(ell + num_io) field operations per proof; the evaluations of 3 run
 * for all proofs in one device pass; the openings of 4 are ONE weighted sum over ipa_gens as in vdfgpu_ipa_verify_batch
 * (comm_E and comm_W are two points of its small MSM, with the scalars -w and -w rho), with its single-proof fallback
 * when the sum is not O.  A proof that fails a host check is left out of both; one that fails 3 is dropped after the
 * opening.  ok_out[q] = 1 iff proof q is valid; the verdicts fail closed: ok_out is zeroed first and receives a 1 only
 * when the whole call succeeded and every check of that proof passed.
 * Verdicts and errors: anything the prover sent is a verdict.  A non-canonical value in the proof record, a
 * non-canonical u or X, or a point with a coordinate >= p or off y^2 = x^3 + 5 gives ok_out[q] = 0 for that proof only
 * and leaves it out of the weighted sum.  VDFGPU_ERR_ARG, before any device work: a null pointer, k = 0, ipa_gens of the
 * wrong curve or with fewer than m + 1 points (U0 = G_m), 1 + num_io > m, a non-canonical value in a challenge record
 * or a weight, an IPA challenge or a weight that is 0.  A sum-check challenge of 0 is legal.
 * Soundness: the weights must be uniform and unpredictable to whoever produced the proofs (the OS CSPRNG, e.g. OsRng);
 * a batch that contains an invalid opening then passes with probability at most 1 / order.  Weights the provers can
 * predict let two invalid openings cancel.  The library never generates weights.  The shape and ipa_gens stay
 * referenced for the whole call, which runs on the calling thread's stream and waits outside the library's lock. */
#define VDFGPU_SPARTAN_PROOF_FES(ell_x) (5 * (ell_x) + 9)
#define VDFGPU_SPARTAN_CHAL_FES(ell_x) (4 * (ell_x) + 6)
#define VDFGPU_SPARTAN_POINTS(ell_x) (2 * (ell_x) + 2)
int vdfgpu_spartan_verify_batch(const vdfgpu_r1cs* s, vdfgpu_gens* ipa_gens, size_t k, const void* inst32_host,
                                const void* points96_host, const void* proof32_host, const void* chal32_host,
                                const void* w32_host, uint8_t* ok_out_host);

/* ---- a8: batched MinRoot verification.  Replaces a loop of MinRootVDF::check (src/minroot.rs:369-371)
 * / Evaluation::verify (:424-426) over independent chains.  ok_out[k] = 1 iff
 * originals[k] == inverse_eval(results[k], t_k).  t_each may be NULL (then every chain uses t_uniform). */
int vdfgpu_minroot_check_batch(int field, const void* results_state96_host,
                               const void* originals_state96_host, const uint64_t* t_each,
                               uint64_t t_uniform, size_t n, uint8_t* ok_out_host);
int vdfgpu_minroot_check_batch_dev(int field, const void* results_dev, const void* originals_dev,
                                   const uint64_t* t_each_dev, uint64_t t_uniform, size_t n,
                                   uint8_t* ok_out_dev);
/* out[k] = inverse_eval(results[k], t): the fast direction, also the step-circuit witness generator */
int vdfgpu_minroot_inverse_eval_batch(int field, const void* results_state96_host, uint64_t t, size_t n,
                                      void* out_state96_host);

/* Step-circuit witness (SURVEY 8f rank 1): for each of n steps, the 4t+1 values InverseMinRootCircuit::synthesize
 * allocates (src/nova/proof.rs:107-126, :162-189) in allocation order: per round new_x, tmp1, tmp2, new_y; then
 * final_i.  out holds n * (4t+1) field elements. */
int vdfgpu_minroot_witness_batch(int field, const void* results_state96_host, uint64_t t, size_t n,
                                 void* out_fe32_host);

/* per-stage device time of the most recent MSM, measured with CUDA events on the stream in use.
 * Stages: 0 digits+histogram, 1 scan, 2 scatter, 3 accumulate, 4 record fix-up, 5 bucket reduction, 6 final */
#define VDFGPU_MSM_STAGES 7
int vdfgpu_profile_enable(int on);
int vdfgpu_profile_read(double* stage_ms, int n_stages);
/* device-pointer variant of vdfgpu_point_sum (multi-GPU combine without a host round trip) */
int vdfgpu_point_sum_dev(int curve, const void* points96_dev, size_t k, void* out_point96_dev);

/* ---- measurement helpers (bench.py) ------------------------------------------------------------------ */
/* elementwise field multiply out[i] = a[i]*b[i] iterated `iters` times (out <- out*b): field-layer parity
 * tests and the integer-multiply roofline probe.  Bit 31 of iters: out-of-line multiplier; bit 30: dedicated
 * squaring instead (out <- out^2, b unused) */
int vdfgpu_field_mul_batch(int field, const void* a_host, const void* b_host, size_t n, uint32_t iters,
                           void* out_host);
/* register-only integer-multiply peak probe: returns 32x32->64 products per second in *out */
int vdfgpu_imad_peak(double* mul32_per_s_wide, double* imad_per_s_lo, double* iadd3_per_s);

#ifdef __cplusplus
}
#endif
#endif /* VDFGPU_H */
