//! src/nova/gpu.rs -- the GPU side of the Nova/MinRoot prover for protocol/vdf, over vdfgpu-sys.
//!
//! NOT COMPILED in the build environment of this repository (no cargo/rustc; dependencies not vendored).  Items
//! marked [R] rely on recalled nova-snark 0.8 / pasta_curves 0.4 APIs and must be checked against the resolved
//! crate versions the first time this is built.
//!
//! What it replaces, all reached today through the single call `RecursiveSNARK::prove_step`
//! (reference src/nova/proof.rs:342-349):
//!   * `GpuGens`      nova `CommitGens` + `commit()` -> `Group::vartime_multiscalar_mul` -> `pasta_msm::{pallas,vesta}`
//!   * `GpuShape`     nova `R1CSShape::{multiply_vec, commit_T}`
//!   * `GpuRunning`   the witness side of `NIFS::prove`: commit(W2), T, commit(T), then
//!                    `RelaxedR1CSWitness::fold` with the challenge -- W and E never leave HBM between steps
//!   * `WitnessBank`  the 4t+1 step-circuit variables of every step (`InverseMinRootCircuit::synthesize`,
//!                    reference src/nova/proof.rs:87-140, :155-230) generated on the device
//!   * `check_batch`  `MinRootVDF::check` (reference src/minroot.rs:369-371) over many independent chains
//!   * `GpuShape::is_sat_relaxed`, `GpuRunning::check`  the satisfiability checks of `RecursiveSNARK::verify`
//!                    (reference src/nova/proof.rs:382): rows and both commitments, `NovaError::UnSat` on failure
//! The public API of the crate (`public_params`, `eval_and_make_circuits`, `NovaVDFProof::{prove_recursively,
//! compress, verify}`) is unchanged; the unmodified nova-snark already reaches the GPU for every commitment through
//! the patched pasta-msm (rust/patches/), and the types below are for a nova-snark whose `NIFS::prove` is patched
//! (or re-implemented in this crate) to keep the running witness on the device.
//!
//! There is no CPU fallback: every constructor fails when no B200 is present.

use std::marker::PhantomData;

use ff::PrimeField;
use nova_snark::errors::NovaError; // [R]: UnSat, InvalidWitnessLength
use pasta_curves::{pallas, vesta};
use vdfgpu_sys as sys;

use crate::minroot::State;

#[derive(Debug)]
pub enum GpuError {
    /// VDFGPU_ERR_ARG: the caller broke the contract (lengths, null handles)
    Argument(String),
    /// VDFGPU_ERR_CUDA: driver / out-of-memory / no device
    Cuda(String),
    /// VDFGPU_ERR_STATE: call order (e.g. fold before commit; destroying generators a running instance still uses)
    State(String),
}

fn check(rc: i32) -> Result<(), GpuError> {
    match rc {
        sys::VDFGPU_OK => Ok(()),
        sys::VDFGPU_ERR_ARG => Err(GpuError::Argument(sys::last_error())),
        sys::VDFGPU_ERR_STATE => Err(GpuError::State(sys::last_error())),
        _ => Err(GpuError::Cuda(sys::last_error())),
    }
}

/// Bind this process to one GPU (one process per GPU; multi-GPU = one process per device, see `sharded_commit`).
pub fn init(device: i32) -> Result<(), GpuError> {
    check(unsafe { sys::vdfgpu_init(device) })
}

/// Curves the library knows, with their `repr-c` types.  Scalars of Pallas are `pallas::Scalar` = Fq, etc.
pub trait GpuCurve {
    const CURVE: i32;
    const SCALAR_FIELD: i32;
    type Affine: Copy;
    type Point: Copy;
    type Scalar: PrimeField;
    fn identity() -> Self::Point;
}
impl GpuCurve for pallas::Point {
    const CURVE: i32 = sys::VDFGPU_PALLAS;
    const SCALAR_FIELD: i32 = sys::VDFGPU_FQ;
    type Affine = pallas::Affine;
    type Point = pallas::Point;
    type Scalar = pallas::Scalar;
    fn identity() -> Self::Point {
        <pallas::Point as group::Group>::identity()
    }
}
impl GpuCurve for vesta::Point {
    const CURVE: i32 = sys::VDFGPU_VESTA;
    const SCALAR_FIELD: i32 = sys::VDFGPU_FP;
    type Affine = vesta::Affine;
    type Point = vesta::Point;
    type Scalar = vesta::Scalar;
    fn identity() -> Self::Point {
        <vesta::Point as group::Group>::identity()
    }
}

/// Device-resident commitment generators: uploaded, repacked (72 -> 64 bytes) and expanded into the 2^(c w) window
/// table ONCE per `PublicParams` (reference src/nova/proof.rs:232-237).
pub struct GpuGens<G: GpuCurve> {
    h: *mut sys::vdfgpu_gens,
    len: usize,
    _g: PhantomData<G>,
}
unsafe impl<G: GpuCurve> Send for GpuGens<G> {}
unsafe impl<G: GpuCurve> Sync for GpuGens<G> {} // the library serialises enqueueing internally

impl<G: GpuCurve> GpuGens<G> {
    /// `raw_jacobian`: commitments come back un-normalised, as pasta-msm's do; `PartialEq`, `to_affine()` and the
    /// transcript code handle that unchanged and the GPU skips one field inversion per commitment.
    pub fn new(gens: &[G::Affine], raw_jacobian: bool) -> Result<Self, GpuError> {
        let mut h = std::ptr::null_mut();
        let flags = sys::VDFGPU_GENS_TABLE | if raw_jacobian { sys::VDFGPU_GENS_RAW_JACOBIAN } else { 0 };
        check(unsafe { sys::vdfgpu_gens_create(G::CURVE, gens.as_ptr().cast(), gens.len(), flags, 0, &mut h) })?;
        Ok(Self { h, len: gens.len(), _g: PhantomData })
    }
    pub fn len(&self) -> usize {
        self.len
    }
    /// nova's `commit`: sum_i scalars[i] * gens[i] over the first `scalars.len()` generators.  Infallible in the
    /// reference (`vartime_multiscalar_mul` returns a point), so a failing GPU call panics like pasta-msm's wrapper.
    pub fn commit(&self, scalars: &[G::Scalar]) -> G::Point {
        assert!(scalars.len() <= self.len, "commit: more scalars than generators");
        let mut out = G::identity();
        let rc = unsafe {
            sys::vdfgpu_msm(self.h, scalars.as_ptr().cast(), scalars.len(), (&mut out as *mut G::Point).cast())
        };
        assert_eq!(rc, 0, "vdfgpu_msm: {}", sys::last_error());
        out
    }
    /// Independent commitments, several in flight: `slot` in 0..4; `scalars` and `out` must stay alive (ideally in
    /// pinned memory) until `commit_wait(slot)` returns.
    pub unsafe fn commit_submit(&self, scalars: &[G::Scalar], out: *mut G::Point, slot: i32) -> Result<(), GpuError> {
        check(sys::vdfgpu_msm_submit(self.h, scalars.as_ptr().cast(), scalars.len(), out.cast(), slot))
    }
    pub fn commit_wait(slot: i32) -> Result<(), GpuError> {
        check(unsafe { sys::vdfgpu_msm_wait(slot) })
    }
}
impl<G: GpuCurve> Drop for GpuGens<G> {
    fn drop(&mut self) {
        unsafe { sys::vdfgpu_gens_destroy(self.h) };
    }
}

/// nova `R1CSShape { A, B, C: Vec<(usize, usize, Scalar)> }` uploaded once as one CSR (column order z = [W | u | X]).
pub struct GpuShape<G: GpuCurve> {
    h: *mut sys::vdfgpu_r1cs,
    pub num_cons: usize,
    pub num_vars: usize,
    pub num_io: usize,
    _g: PhantomData<G>,
}

unsafe impl<G: GpuCurve> Send for GpuShape<G> {}
unsafe impl<G: GpuCurve> Sync for GpuShape<G> {} // read-only after creation; verify checks from several threads

fn split_coo<F: Copy>(m: &[(usize, usize, F)]) -> (Vec<u64>, Vec<u64>, Vec<F>) {
    (m.iter().map(|e| e.0 as u64).collect(), m.iter().map(|e| e.1 as u64).collect(), m.iter().map(|e| e.2).collect())
}

impl<G: GpuCurve> GpuShape<G> {
    pub fn new(
        num_cons: usize,
        num_vars: usize,
        num_io: usize,
        a: &[(usize, usize, G::Scalar)],
        b: &[(usize, usize, G::Scalar)],
        c: &[(usize, usize, G::Scalar)],
    ) -> Result<Self, GpuError> {
        let (ar, ac, av) = split_coo(a);
        let (br, bc, bv) = split_coo(b);
        let (cr, cc, cv) = split_coo(c);
        let mut h = std::ptr::null_mut();
        check(unsafe {
            sys::vdfgpu_r1cs_create(
                G::SCALAR_FIELD, num_cons, num_vars, num_io,
                ar.as_ptr(), ac.as_ptr(), av.as_ptr().cast(), av.len(),
                br.as_ptr(), bc.as_ptr(), bv.as_ptr().cast(), bv.len(),
                cr.as_ptr(), cc.as_ptr(), cv.as_ptr().cast(), cv.len(),
                &mut h,
            )
        })?;
        Ok(Self { h, num_cons, num_vars, num_io, _g: PhantomData })
    }
    /// `R1CSShape::multiply_vec(z)`; nova returns `NovaError::InvalidWitnessLength` on a wrong length.
    pub fn multiply_vec(&self, z: &[G::Scalar]) -> Result<(Vec<G::Scalar>, Vec<G::Scalar>, Vec<G::Scalar>), GpuError> {
        if z.len() != self.num_vars + 1 + self.num_io {
            return Err(GpuError::Argument("InvalidWitnessLength".into()));
        }
        let zero = <G::Scalar as ff::Field>::zero();
        let (mut az, mut bz, mut cz) = (vec![zero; self.num_cons], vec![zero; self.num_cons], vec![zero; self.num_cons]);
        check(unsafe {
            sys::vdfgpu_multiply_vec(self.h, z.as_ptr().cast(), az.as_mut_ptr().cast(), bz.as_mut_ptr().cast(), cz.as_mut_ptr().cast())
        })?;
        Ok((az, bz, cz))
    }
    /// `RelaxedR1CSShape::is_sat_relaxed(gens, U, W)` [R] with the vectors on the host: `e = None` is E = 0 and
    /// `u = None` is u = 1 (both `None`: `R1CSShape::is_sat` of a fresh instance).  `NovaError::UnSat` when a row or a
    /// given commitment does not check out; a commitment that is `None` is not checked.  Infallible otherwise, like
    /// nova's (a failing GPU call panics).
    #[allow(clippy::too_many_arguments)]
    pub fn is_sat_relaxed(
        &self,
        gens: &GpuGens<G>,
        w: &[G::Scalar],
        e: Option<&[G::Scalar]>,
        u: Option<&G::Scalar>,
        x: &[G::Scalar],
        comm_w: Option<&G::Point>,
        comm_e: Option<&G::Point>,
    ) -> Result<(), NovaError> {
        if w.len() != self.num_vars || x.len() != self.num_io || e.map_or(false, |e| e.len() != self.num_cons) {
            return Err(NovaError::InvalidWitnessLength);
        }
        let mut rep = [0u64; 4];
        let rc = unsafe {
            sys::vdfgpu_r1cs_is_sat_relaxed(
                self.h, gens.h, w.as_ptr().cast(), e.map_or(std::ptr::null(), |e| e.as_ptr().cast()),
                u.map_or(std::ptr::null(), |u| (u as *const G::Scalar).cast()), x.as_ptr().cast(),
                point_ptr::<G>(comm_w), point_ptr::<G>(comm_e), rep.as_mut_ptr(),
            )
        };
        assert_eq!(rc, 0, "vdfgpu_r1cs_is_sat_relaxed: {}", sys::last_error());
        sat_verdict(&rep)
    }
}

fn point_ptr<G: GpuCurve>(p: Option<&G::Point>) -> *const libc::c_void {
    p.map_or(std::ptr::null(), |p| (p as *const G::Point).cast())
}

/// report = [violating rows, first violating row, comm_W check, comm_E check] (1 equal, 0 different, 2 not checked)
fn sat_verdict(rep: &[u64; 4]) -> Result<(), NovaError> {
    if rep[0] == 0 && rep[2] != 0 && rep[3] != 0 {
        Ok(())
    } else {
        Err(NovaError::UnSat)
    }
}

impl<G: GpuCurve> Drop for GpuShape<G> {
    fn drop(&mut self) {
        unsafe { sys::vdfgpu_r1cs_destroy(self.h) };
    }
}

/// Step-circuit witnesses of all steps of one proof, generated and kept on the device (SURVEY 8f rank 1).
/// `z_in[k]` is the input state of step k's circuit, i.e. `circuits[k].result` in `prove_recursively`
/// (reference src/nova/proof.rs:318-349); the circuits are independent once the VDF states are known (:284-296).
pub struct WitnessBank<G: GpuCurve> {
    h: *mut sys::vdfgpu_witness_bank,
    pub t: u64,
    _g: PhantomData<G>,
}
impl<G: GpuCurve> WitnessBank<G> {
    pub fn new(z_in: &[State<G::Scalar>], t: u64) -> Result<Self, GpuError> {
        // State<T> is { x, y, i }; it needs #[repr(C)] in src/minroot.rs:267-272 for this cast to be defined
        let mut h = std::ptr::null_mut();
        check(unsafe { sys::vdfgpu_witness_bank_create(G::SCALAR_FIELD, z_in.as_ptr().cast(), t, z_in.len(), &mut h) })?;
        Ok(Self { h, t, _g: PhantomData })
    }
}
impl<G: GpuCurve> Drop for WitnessBank<G> {
    fn drop(&mut self) {
        unsafe { sys::vdfgpu_witness_bank_destroy(self.h) };
    }
}

/// The running relaxed witness (W, E) and instance scalars (u, X) of one curve, resident on the device.
/// One fold step = `commit` (returns what the random oracle absorbs) then `fold` (with the challenge it squeezed).
pub struct GpuRunning<'a, G: GpuCurve> {
    h: *mut sys::vdfgpu_running,
    shape: &'a GpuShape<G>,
    _gens: &'a GpuGens<G>,
}
impl<'a, G: GpuCurve> GpuRunning<'a, G> {
    pub fn new(shape: &'a GpuShape<G>, gens: &'a GpuGens<G>) -> Result<Self, GpuError> {
        let mut h = std::ptr::null_mut();
        check(unsafe { sys::vdfgpu_running_create(shape.h, gens.h, &mut h) })?;
        Ok(Self { h, shape, _gens: gens })
    }
    /// Load a running instance (after the base case: W = W_1, E = 0, u = 1, X = X_1).
    pub fn set(&mut self, w: &[G::Scalar], e: &[G::Scalar], u: &G::Scalar, x: &[G::Scalar]) -> Result<(), GpuError> {
        if w.len() != self.shape.num_vars || e.len() != self.shape.num_cons || x.len() != self.shape.num_io {
            return Err(GpuError::Argument("InvalidWitnessLength".into()));
        }
        check(unsafe {
            sys::vdfgpu_running_set(self.h, w.as_ptr().cast(), e.as_ptr().cast(), (u as *const G::Scalar).cast(), x.as_ptr().cast())
        })
    }
    /// commit(W2), T = Az1.Bz2 + Az2.Bz1 - u1.Cz2 - Cz1, commit(T): ONE batched MSM over the shared generators.
    pub fn commit(&mut self, w2: &[G::Scalar], x2: &[G::Scalar]) -> Result<(G::Point, G::Point), GpuError> {
        if w2.len() != self.shape.num_vars || x2.len() != self.shape.num_io {
            return Err(GpuError::Argument("InvalidWitnessLength".into()));
        }
        let (mut cw, mut ct) = (G::identity(), G::identity());
        check(unsafe {
            sys::vdfgpu_running_commit(self.h, w2.as_ptr().cast(), x2.as_ptr().cast(),
                                       (&mut cw as *mut G::Point).cast(), (&mut ct as *mut G::Point).cast())
        })?;
        Ok((cw, ct))
    }
    /// `commit` with W2[step_offset .. step_offset + 4t + 1] taken from the bank: those entries of `w2` are ignored.
    pub fn commit_step(&mut self, bank: &WitnessBank<G>, step: usize, step_offset: usize, w2: &[G::Scalar],
                       x2: &[G::Scalar]) -> Result<(G::Point, G::Point), GpuError> {
        if w2.len() != self.shape.num_vars || x2.len() != self.shape.num_io {
            return Err(GpuError::Argument("InvalidWitnessLength".into()));
        }
        let (mut cw, mut ct) = (G::identity(), G::identity());
        check(unsafe {
            sys::vdfgpu_running_commit_step(self.h, bank.h, step, step_offset, w2.as_ptr().cast(), x2.as_ptr().cast(),
                                            (&mut cw as *mut G::Point).cast(), (&mut ct as *mut G::Point).cast())
        })?;
        Ok((cw, ct))
    }
    /// `RelaxedR1CSWitness::fold` + the scalar half of `RelaxedR1CSInstance::fold`:
    /// W += r W2, E += r T, u += r, X += r X2.  Returns at once; the next call on this instance is ordered behind it
    /// on the GPU, whichever stream (`vdfgpu_set_stream`) or thread it comes from: a verifier thread may `check` it.
    pub fn fold(&mut self, r: &G::Scalar) -> Result<(), GpuError> {
        check(unsafe { sys::vdfgpu_running_finish(self.h, (r as *const G::Scalar).cast()) })
    }
    /// Read the running witness back (needed by `CompressedSNARK::prove` only; `check` verifies it in place).
    pub fn get(&self) -> Result<(Vec<G::Scalar>, Vec<G::Scalar>, G::Scalar, Vec<G::Scalar>), GpuError> {
        let zero = <G::Scalar as ff::Field>::zero();
        let (mut w, mut e, mut u, mut x) =
            (vec![zero; self.shape.num_vars], vec![zero; self.shape.num_cons], zero, vec![zero; self.shape.num_io]);
        check(unsafe {
            sys::vdfgpu_running_get(self.h, w.as_mut_ptr().cast(), e.as_mut_ptr().cast(),
                                    (&mut u as *mut G::Scalar).cast(), x.as_mut_ptr().cast())
        })?;
        Ok((w, e, u, x))
    }
    /// `is_sat_relaxed` of the resident running instance against the instance's commitments (`U.comm_W`, `U.comm_E`):
    /// the relaxed half of `RecursiveSNARK::verify` without copying W and E back.  `NovaError::UnSat` on a failed check.
    pub fn check(&self, comm_w: Option<&G::Point>, comm_e: Option<&G::Point>) -> Result<(), NovaError> {
        let mut rep = [0u64; 4];
        let rc = unsafe { sys::vdfgpu_running_check(self.h, point_ptr::<G>(comm_w), point_ptr::<G>(comm_e), rep.as_mut_ptr()) };
        assert_eq!(rc, 0, "vdfgpu_running_check: {}", sys::last_error());
        sat_verdict(&rep)
    }
}
impl<'a, G: GpuCurve> Drop for GpuRunning<'a, G> {
    fn drop(&mut self) {
        unsafe { sys::vdfgpu_running_destroy(self.h) };
    }
}

/// One `NIFS::prove` with the running witness on the device [R: nova-snark 0.8 nifs.rs].  `ro_challenge` is nova's
/// Poseidon random oracle over (params, U1, U2, comm_T), untouched and on the host; the instance-side commitment
/// folds (two scalar multiplications) stay where they are in `RelaxedR1CSInstance::fold`.
pub fn nifs_prove_witness<G: GpuCurve>(
    run: &mut GpuRunning<'_, G>,
    w2: &[G::Scalar],
    x2: &[G::Scalar],
    ro_challenge: impl FnOnce(&G::Point, &G::Point) -> G::Scalar,
) -> Result<(G::Point, G::Point, G::Scalar), GpuError> {
    let (comm_w2, comm_t) = run.commit(w2, x2)?;
    let r = ro_challenge(&comm_w2, &comm_t);
    run.fold(&r)?;
    Ok((comm_w2, comm_t, r))
}

/// `MinRootVDF::check` (reference src/minroot.rs:369-371) for many independent (result, t, original) triples;
/// `Evaluation::verify` / `append` (:424-438) over many segments are batches of the same call.
pub fn check_batch<G: GpuCurve>(results: &[State<G::Scalar>], ts: &[u64], originals: &[State<G::Scalar>]) -> Vec<bool> {
    assert!(results.len() == ts.len() && ts.len() == originals.len());
    let mut ok = vec![0u8; results.len()];
    let rc = unsafe {
        sys::vdfgpu_minroot_check_batch(G::SCALAR_FIELD, results.as_ptr().cast(), originals.as_ptr().cast(), ts.as_ptr(), 0,
                                        results.len(), ok.as_mut_ptr())
    };
    assert_eq!(rc, 0, "vdfgpu_minroot_check_batch: {}", sys::last_error());
    ok.into_iter().map(|b| b != 0).collect()
}

/// Multi-GPU commitment (one process per GPU): this rank commits its contiguous slice with its own `GpuGens`
/// (created with `raw_jacobian = true`), `exchange` all-gathers the 96-byte partial points over whatever transport
/// the deployment has (NCCL, MPI), and one warp on the GPU adds them and normalises once.
pub fn sharded_commit<G: GpuCurve>(
    gens_slice: &GpuGens<G>,
    scalars_slice: &[G::Scalar],
    exchange: impl FnOnce(&G::Point) -> Vec<G::Point>,
) -> G::Point {
    let part = gens_slice.commit(scalars_slice);
    let parts = exchange(&part);
    let mut out = G::identity();
    let rc = unsafe { sys::vdfgpu_point_sum(G::CURVE, parts.as_ptr().cast(), parts.len(), (&mut out as *mut G::Point).cast()) };
    assert_eq!(rc, 0, "vdfgpu_point_sum: {}", sys::last_error());
    out
}
