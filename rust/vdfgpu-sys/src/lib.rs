//! Raw FFI bindings to libvdfgpu (include/vdfgpu.h), one declaration per exported symbol.
//!
//! NOT COMPILED in the build environment of this repository (no cargo/rustc there); kept in step with the header by
//! tests/test_rust_bindings.py.  Layouts: pasta_curves with feature `repr-c` (reference Cargo.toml:17) --
//! field element 32 B (four LE u64 limbs, Montgomery), affine point 72 B, Jacobian point 96 B, State<F> 96 B.
#![allow(non_camel_case_types)]

use libc::{c_char, c_int, c_void, size_t};

pub const VDFGPU_PALLAS: c_int = 0;
pub const VDFGPU_VESTA: c_int = 1;
pub const VDFGPU_FP: c_int = 0;
pub const VDFGPU_FQ: c_int = 1;

pub const VDFGPU_OK: c_int = 0;
pub const VDFGPU_ERR_ARG: c_int = -1;
pub const VDFGPU_ERR_CUDA: c_int = -2;
pub const VDFGPU_ERR_STATE: c_int = -3;

pub const VDFGPU_GENS_TABLE: u32 = 1;
pub const VDFGPU_GENS_RAW_JACOBIAN: u32 = 2;
pub const VDFGPU_MSM_STAGES: c_int = 7;

#[repr(C)]
pub struct vdfgpu_gens {
    _private: [u8; 0],
}
#[repr(C)]
pub struct vdfgpu_r1cs {
    _private: [u8; 0],
}
#[repr(C)]
pub struct vdfgpu_running {
    _private: [u8; 0],
}
#[repr(C)]
pub struct vdfgpu_witness_bank {
    _private: [u8; 0],
}

/// Per-round callback of the sum-check drivers: receives the round's evaluations (n_evals field elements), owns the
/// transcript, writes the challenge to `r_out_fe32`, returns 0.
pub type vdfgpu_round_fn = Option<
    unsafe extern "C" fn(user: *mut c_void, round: size_t, evals_fe32: *const c_void, n_evals: size_t, r_out_fe32: *mut c_void) -> c_int,
>;

/// Per-round callback of the inner-product argument: receives the round's commitments L and R (96-byte normalised
/// points, identity = 96 zero bytes), owns the transcript, writes the challenge r != 0 to `r_out32`, returns 0.
pub type vdfgpu_ipa_round_fn = Option<
    unsafe extern "C" fn(user: *mut c_void, round: size_t, l_point96: *const c_void, r_point96: *const c_void, r_out32: *mut c_void) -> c_int,
>;

/// Claims callback of `vdfgpu_running_spartan_prove`: at stage OUTER receives (claim_Az, claim_Bz, claim_Cz, eval_E) and
/// writes (r_A, r_B, r_C); at EVAL receives (eval_W, T) and writes rho; at IPA receives c and writes u_scale; returns 0.
pub type vdfgpu_spartan_claims_fn = Option<
    unsafe extern "C" fn(user: *mut c_void, stage: c_int, in_fe32: *const c_void, n_in: size_t, out_fe32: *mut c_void,
                         n_out: size_t) -> c_int,
>;
pub const VDFGPU_SPARTAN_OUTER: c_int = 0;
pub const VDFGPU_SPARTAN_EVAL: c_int = 1;
pub const VDFGPU_SPARTAN_IPA: c_int = 2;

extern "C" {
    // ---- context
    pub fn vdfgpu_init(device: c_int) -> c_int;
    pub fn vdfgpu_shutdown() -> c_int;
    pub fn vdfgpu_device_count() -> c_int;
    pub fn vdfgpu_last_error() -> *const c_char;
    pub fn vdfgpu_version() -> *const c_char;
    pub fn vdfgpu_set_stream(cuda_stream: *mut c_void) -> c_int;
    pub fn vdfgpu_synchronize() -> c_int;
    pub fn vdfgpu_trim() -> c_int;
    pub fn vdfgpu_launch_count() -> u64;

    // ---- a4: MSM.  The first two are pasta-msm's own symbols (its wrapper binds them itself).
    pub fn mult_pippenger_pallas(out_point96: *mut c_void, points_affine72: *const c_void, npoints: size_t,
                                 scalars32: *const c_void, is_mont: bool);
    pub fn mult_pippenger_vesta(out_point96: *mut c_void, points_affine72: *const c_void, npoints: size_t,
                                scalars32: *const c_void, is_mont: bool);
    pub fn vdfgpu_dropin_cache_clear() -> c_int;
    pub fn vdfgpu_dropin_cache_stats(hits: *mut u64, misses: *mut u64, entries: *mut u64) -> c_int;

    pub fn vdfgpu_gens_create(curve: c_int, points_affine72_host: *const c_void, n: size_t, flags: u32,
                              window_bits: u32, out: *mut *mut vdfgpu_gens) -> c_int;
    pub fn vdfgpu_gens_progression(curve: c_int, k0_le32: *const c_void, d_le32: *const c_void, n: size_t, flags: u32,
                                   window_bits: u32, out: *mut *mut vdfgpu_gens) -> c_int;
    pub fn vdfgpu_gens_export(g: *const vdfgpu_gens, first: size_t, count: size_t,
                              points_affine72_host: *mut c_void) -> c_int;
    pub fn vdfgpu_gens_len(g: *const vdfgpu_gens) -> size_t;
    pub fn vdfgpu_gens_window_bits(g: *const vdfgpu_gens, n: size_t) -> u32;
    pub fn vdfgpu_gens_affine_rounds(g: *const vdfgpu_gens, n: size_t) -> u32;
    pub fn vdfgpu_gens_destroy(g: *mut vdfgpu_gens) -> c_int;

    pub fn vdfgpu_msm(g: *mut vdfgpu_gens, scalars32_host: *const c_void, n: size_t,
                      out_point96_host: *mut c_void) -> c_int;
    pub fn vdfgpu_msm_dev(g: *mut vdfgpu_gens, scalars32_dev: *const c_void, n: size_t,
                          out_point96_dev: *mut c_void) -> c_int;
    pub fn vdfgpu_msm_submit(g: *mut vdfgpu_gens, scalars32_host: *const c_void, n: size_t,
                             out_point96_host: *mut c_void, slot: c_int) -> c_int;
    pub fn vdfgpu_msm_wait(slot: c_int) -> c_int;
    pub fn vdfgpu_msm_batch_dev(g: *mut vdfgpu_gens, scalars32_dev: *const *const c_void, lens: *const size_t, k: u32,
                                out_points96_dev: *mut c_void) -> c_int;
    pub fn vdfgpu_msm_range_dev(g: *mut vdfgpu_gens, first: size_t, scalars32_dev: *const c_void, n: size_t,
                                out_point96_dev: *mut c_void) -> c_int;
    pub fn vdfgpu_point_normalise_host(curve: c_int, points96_host: *mut c_void, count: size_t) -> c_int;
    pub fn vdfgpu_point_sum(curve: c_int, points96_host: *const c_void, k: size_t,
                            out_point96_host: *mut c_void) -> c_int;
    pub fn vdfgpu_point_sum_dev(curve: c_int, points96_dev: *const c_void, k: size_t,
                                out_point96_dev: *mut c_void) -> c_int;

    // ---- a5-a7: R1CS
    pub fn vdfgpu_r1cs_create(field: c_int, num_cons: size_t, num_vars: size_t, num_io: size_t,
                              a_rows: *const u64, a_cols: *const u64, a_vals32: *const c_void, a_nnz: size_t,
                              b_rows: *const u64, b_cols: *const u64, b_vals32: *const c_void, b_nnz: size_t,
                              c_rows: *const u64, c_cols: *const u64, c_vals32: *const c_void, c_nnz: size_t,
                              out: *mut *mut vdfgpu_r1cs) -> c_int;
    pub fn vdfgpu_r1cs_destroy(s: *mut vdfgpu_r1cs) -> c_int;
    pub fn vdfgpu_multiply_vec(s: *const vdfgpu_r1cs, z_host: *const c_void, az_host: *mut c_void,
                               bz_host: *mut c_void, cz_host: *mut c_void) -> c_int;
    pub fn vdfgpu_commit_T(s: *const vdfgpu_r1cs, gens: *mut vdfgpu_gens, w1_host: *const c_void,
                           u1_host: *const c_void, x1_host: *const c_void, w2_host: *const c_void,
                           x2_host: *const c_void, t_host: *mut c_void, comm_t_point96_host: *mut c_void) -> c_int;
    pub fn vdfgpu_fold(field: c_int, w1_host: *mut c_void, w2_host: *const c_void, n_w: size_t, e1_host: *mut c_void,
                       t_host: *const c_void, n_e: size_t, r32_host: *const c_void) -> c_int;
    pub fn vdfgpu_multiply_vec_dev(s: *const vdfgpu_r1cs, w_dev: *const c_void, ux_dev: *const c_void,
                                   az_bz_cz_dev: *mut c_void) -> c_int;
    pub fn vdfgpu_r1cs_bind_rows(s: *const vdfgpu_r1cs, eq_rows_host: *const c_void, r_abc_host: *const c_void,
                                 out_host: *mut c_void) -> c_int;
    pub fn vdfgpu_r1cs_bind_rows_dev(s: *const vdfgpu_r1cs, eq_rows_dev: *const c_void, r_abc_dev: *const c_void,
                                     scratch_dev: *mut c_void, out_dev: *mut c_void) -> c_int;
    pub fn vdfgpu_cross_term_dev(s: *const vdfgpu_r1cs, w1_dev: *const c_void, ux1_dev: *const c_void,
                                 w2_dev: *const c_void, ux2_dev: *const c_void, t_dev: *mut c_void) -> c_int;
    pub fn vdfgpu_fold_dev(field: c_int, w1_dev: *mut c_void, w2_dev: *const c_void, n_w: size_t, e1_dev: *mut c_void,
                           t_dev: *const c_void, n_e: size_t, r32_dev: *const c_void) -> c_int;

    pub fn vdfgpu_running_create(s: *const vdfgpu_r1cs, gens: *mut vdfgpu_gens, out: *mut *mut vdfgpu_running) -> c_int;
    pub fn vdfgpu_running_destroy(f: *mut vdfgpu_running) -> c_int;
    pub fn vdfgpu_running_set(f: *mut vdfgpu_running, w_host: *const c_void, e_host: *const c_void,
                              u_host: *const c_void, x_host: *const c_void) -> c_int;
    pub fn vdfgpu_running_get(f: *const vdfgpu_running, w_host: *mut c_void, e_host: *mut c_void, u_host: *mut c_void,
                              x_host: *mut c_void) -> c_int;
    pub fn vdfgpu_running_commit(f: *mut vdfgpu_running, w2_host: *const c_void, x2_host: *const c_void,
                                 comm_w2_point96_host: *mut c_void, comm_t_point96_host: *mut c_void) -> c_int;
    pub fn vdfgpu_running_finish(f: *mut vdfgpu_running, r32_host: *const c_void) -> c_int;

    // ---- RecursiveSNARK::verify: is_sat_relaxed / is_sat; report = [bad rows, first bad row, comm_W ok, comm_E ok]
    pub fn vdfgpu_r1cs_is_sat_relaxed(s: *const vdfgpu_r1cs, gens: *mut vdfgpu_gens, w_host: *const c_void,
                                      e_host: *const c_void, u_host: *const c_void, x_host: *const c_void,
                                      comm_w96_host: *const c_void, comm_e96_host: *const c_void,
                                      report4_host: *mut u64) -> c_int;
    pub fn vdfgpu_r1cs_is_sat_relaxed_dev(s: *const vdfgpu_r1cs, w_dev: *const c_void, e_dev: *const c_void,
                                          ux_dev: *const c_void, counts2_dev: *mut u64) -> c_int;
    pub fn vdfgpu_running_check(f: *const vdfgpu_running, comm_w96_host: *const c_void, comm_e96_host: *const c_void,
                                report4_host: *mut u64) -> c_int;

    // ---- SURVEY 8f rank 1: step-circuit witnesses generated and kept on the device
    pub fn vdfgpu_witness_bank_create(field: c_int, z_in_state96_host: *const c_void, t: u64, n: size_t,
                                      out: *mut *mut vdfgpu_witness_bank) -> c_int;
    pub fn vdfgpu_witness_bank_destroy(b: *mut vdfgpu_witness_bank) -> c_int;
    pub fn vdfgpu_witness_bank_read(b: *const vdfgpu_witness_bank, first_step: size_t, count: size_t,
                                    out_fe32_host: *mut c_void) -> c_int;
    pub fn vdfgpu_running_commit_step(f: *mut vdfgpu_running, bank: *const vdfgpu_witness_bank, step: size_t,
                                      step_offset: size_t, w2_host: *const c_void, x2_host: *const c_void,
                                      comm_w2_point96_host: *mut c_void, comm_t_point96_host: *mut c_void) -> c_int;

    // ---- SURVEY 8f rank 2: sum-check building blocks (CompressedSNARK::prove)
    pub fn vdfgpu_eq_evals(field: c_int, r_host: *const c_void, ell: size_t, out_host: *mut c_void) -> c_int;
    pub fn vdfgpu_eq_evals_dev(field: c_int, r_host: *const c_void, ell: size_t, out_dev: *mut c_void) -> c_int;
    pub fn vdfgpu_sumcheck_cubic(field: c_int, a_host: *const c_void, b_host: *const c_void, c_host: *const c_void,
                                 d_host: *const c_void, ell: size_t, round_fn: vdfgpu_round_fn, user: *mut c_void,
                                 final_evals4_host: *mut c_void) -> c_int;
    pub fn vdfgpu_sumcheck_cubic_dev(field: c_int, a_dev: *mut c_void, b_dev: *mut c_void, c_dev: *mut c_void,
                                     d_dev: *mut c_void, ell: size_t, round_fn: vdfgpu_round_fn, user: *mut c_void,
                                     final_evals4_host: *mut c_void) -> c_int;
    pub fn vdfgpu_sumcheck_quad(field: c_int, a_host: *const c_void, b_host: *const c_void, ell: size_t,
                                round_fn: vdfgpu_round_fn, user: *mut c_void, final_evals2_host: *mut c_void) -> c_int;
    pub fn vdfgpu_sumcheck_quad_dev(field: c_int, a_dev: *mut c_void, b_dev: *mut c_void, ell: size_t,
                                    round_fn: vdfgpu_round_fn, user: *mut c_void, final_evals2_host: *mut c_void) -> c_int;
    pub fn vdfgpu_poly_evaluate(field: c_int, poly_host: *const c_void, r_host: *const c_void, ell: size_t,
                                out_host: *mut c_void) -> c_int;
    pub fn vdfgpu_poly_evaluate_dev(field: c_int, poly_dev: *const c_void, r_host: *const c_void, ell: size_t,
                                    out_host: *mut c_void) -> c_int;

    pub fn vdfgpu_vec_lincomb(field: c_int, a_host: *const c_void, b_host: *const c_void, n: size_t, x32_host: *const c_void,
                              y32_host: *const c_void, out_host: *mut c_void) -> c_int;
    pub fn vdfgpu_inner_product(field: c_int, a_host: *const c_void, b_host: *const c_void, n: size_t,
                                out32_host: *mut c_void) -> c_int;
    pub fn vdfgpu_points_lincomb(curve: c_int, p_affine72_host: *const c_void, q_affine72_host: *const c_void, n: size_t,
                                 w1_32_host: *const c_void, w2_32_host: *const c_void, out_affine72_host: *mut c_void) -> c_int;
    pub fn vdfgpu_ipa_prove(g: *mut vdfgpu_gens, a_host: *const c_void, b_host: *const c_void, ell: size_t,
                            u_scale32_host: *const c_void, round_fn: vdfgpu_ipa_round_fn, user: *mut c_void,
                            a_hat32_host: *mut c_void) -> c_int;
    pub fn vdfgpu_ipa_prove_dev(g: *mut vdfgpu_gens, a_dev: *mut c_void, b_dev: *mut c_void, ell: size_t,
                                u_scale32_host: *const c_void, round_fn: vdfgpu_ipa_round_fn, user: *mut c_void,
                                a_hat32_host: *mut c_void) -> c_int;
    pub fn vdfgpu_ipa_gens_hat(g: *mut vdfgpu_gens, r_host: *const c_void, ell: size_t, out_point96_host: *mut c_void) -> c_int;
    pub fn vdfgpu_ipa_verify_batch(g: *mut vdfgpu_gens, ell: size_t, k: size_t, comm_a96_host: *const c_void,
                                   l96_host: *const c_void, r96_host: *const c_void, r32_host: *const c_void,
                                   a_hat32_host: *const c_void, c32_host: *const c_void, b_hat32_host: *const c_void,
                                   u_scale32_host: *const c_void, w32_host: *const c_void, ok_out_host: *mut u8) -> c_int;

    // ---- RelaxedR1CSSNARK::prove of the running instance in one call, and the verifier's sparse evaluation
    pub fn vdfgpu_running_spartan_prove(f: *mut vdfgpu_running, ipa_gens: *mut vdfgpu_gens, tau_host: *const c_void,
                                        sc_round: vdfgpu_round_fn, claims: vdfgpu_spartan_claims_fn,
                                        ipa_round: vdfgpu_ipa_round_fn, user: *mut c_void,
                                        a_hat32_host: *mut c_void) -> c_int;
    pub fn vdfgpu_r1cs_evaluate(s: *const vdfgpu_r1cs, rx_host: *const c_void, ry_host: *const c_void,
                                out3_host: *mut c_void) -> c_int;
    pub fn vdfgpu_r1cs_evaluate_batch(s: *const vdfgpu_r1cs, k: size_t, rx_host: *const c_void, ry_host: *const c_void,
                                      out3_host: *mut c_void) -> c_int;
    pub fn vdfgpu_spartan_verify_batch(s: *const vdfgpu_r1cs, ipa_gens: *mut vdfgpu_gens, k: size_t,
                                       inst32_host: *const c_void, points96_host: *const c_void,
                                       proof32_host: *const c_void, chal32_host: *const c_void,
                                       w32_host: *const c_void, ok_out_host: *mut u8) -> c_int;

    // ---- a8: batched MinRoot verification
    pub fn vdfgpu_minroot_check_batch(field: c_int, results_state96_host: *const c_void,
                                      originals_state96_host: *const c_void, t_each: *const u64, t_uniform: u64,
                                      n: size_t, ok_out_host: *mut u8) -> c_int;
    pub fn vdfgpu_minroot_check_batch_dev(field: c_int, results_dev: *const c_void, originals_dev: *const c_void,
                                          t_each_dev: *const u64, t_uniform: u64, n: size_t, ok_out_dev: *mut u8) -> c_int;
    pub fn vdfgpu_minroot_inverse_eval_batch(field: c_int, results_state96_host: *const c_void, t: u64, n: size_t,
                                             out_state96_host: *mut c_void) -> c_int;
    pub fn vdfgpu_minroot_witness_batch(field: c_int, results_state96_host: *const c_void, t: u64, n: size_t,
                                        out_fe32_host: *mut c_void) -> c_int;

    // ---- measurement helpers
    pub fn vdfgpu_profile_enable(on: c_int) -> c_int;
    pub fn vdfgpu_profile_read(stage_ms: *mut f64, n_stages: c_int) -> c_int;
    pub fn vdfgpu_field_mul_batch(field: c_int, a_host: *const c_void, b_host: *const c_void, n: size_t, iters: u32,
                                  out_host: *mut c_void) -> c_int;
    pub fn vdfgpu_imad_peak(mul32_per_s_wide: *mut f64, imad_per_s_lo: *mut f64, iadd3_per_s: *mut f64) -> c_int;
}

/// Thread-local message of the last failing call on this thread.
pub fn last_error() -> String {
    unsafe {
        let p = vdfgpu_last_error();
        if p.is_null() {
            String::new()
        } else {
            std::ffi::CStr::from_ptr(p).to_string_lossy().into_owned()
        }
    }
}
