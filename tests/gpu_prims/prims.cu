// Test harness: the library's device primitives one operation at a time (tests/test_gpu_primitives.py).
//
// Like tests/emul/emul.cpp this is a test tool, never linked into libvdfgpu.so.  It includes the library headers
// unchanged and runs their DEVICE branches -- the PTX carry chains of field.cuh, the XYZZ group law of curve.cuh as
// compiled for sm_100a, the four-lane group law of quad.cuh (which has no host version) and the batched-affine
// functors of msm_affine.cuh -- elementwise on caller arrays, so that Python integers can check each result.
//
// Every entry point copies its inputs to the device, runs one small grid, copies the results back, frees everything
// and returns 0, or the CUDA error code.  Field elements are raw 32-byte Montgomery limbs; `field` / `curve` is 0 for
// Fp / Pallas and 1 for Fq / Vesta.
#include <cuda_runtime.h>

#include <cstdint>
#include <cstring>
#include <stdexcept>
#include <vector>

#include "../../vdf_b200/csrc/msm_affine.cuh"
#include "../../vdf_b200/csrc/quad.cuh"

using namespace vdf;

namespace {

// ---- field: one kernel per operation -------------------------------------------------------------
enum FieldOp {
  F_ADD = 0, F_SUB, F_NEG, F_DBL, F_MUL, F_MUL_CALL, F_MUL_VAL, F_SQR, F_SQR_CALL, F_SQR_VAL,
  F_FROM_MONT, F_INV, F_ONE, F_IS_CANONICAL, F_EQ, F_IS_ZERO, F_NOPS
};

template <class F, int OP>
__global__ void field_kernel(const fe* a, const fe* b, fe* out, uint8_t* flag, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const fe x = fe_load(a + i), y = fe_load(b + i);
  fe r = F::zero();
  if constexpr (OP == F_ADD) r = F::add(x, y);
  else if constexpr (OP == F_SUB) r = F::sub(x, y);
  else if constexpr (OP == F_NEG) r = F::neg(x);
  else if constexpr (OP == F_DBL) r = F::dbl(x);
  else if constexpr (OP == F_MUL) r = F::mul(x, y);
  else if constexpr (OP == F_MUL_CALL) r = F::mul_call(x, y);
  else if constexpr (OP == F_MUL_VAL) r = F::mul_val(x, y);
  else if constexpr (OP == F_SQR) r = F::sqr(x);
  else if constexpr (OP == F_SQR_CALL) r = F::sqr_call(x);
  else if constexpr (OP == F_SQR_VAL) r = F::sqr_val(x);
  else if constexpr (OP == F_FROM_MONT) r = F::from_mont(x);
  else if constexpr (OP == F_INV) r = F::inv(x);
  else if constexpr (OP == F_ONE) r = F::one();
  else if constexpr (OP == F_IS_CANONICAL) { flag[i] = F::is_canonical(x); return; }
  else if constexpr (OP == F_EQ) { flag[i] = F::eq(x, y); return; }
  else if constexpr (OP == F_IS_ZERO) { flag[i] = F::is_zero(x); return; }
  fe_store(out + i, r);
}

// ---- curve: elementwise on XYZZ / affine / Jacobian arrays -----------------------------------------
enum CurveOp {
  C_FROM_AFFINE = 0,   // a: affine           -> xyzz
  C_MADD,              // a: xyzz, b: affine  -> xyzz  (operand not the identity)
  C_MADD_CALL,
  C_MADD_SIGNED,       // a: xyzz, b: affine, aux: negate -> xyzz
  C_MADD_SIGNED_CALL,
  C_DBL_AFFINE,        // a: affine           -> xyzz
  C_DBL,               // a: xyzz             -> xyzz
  C_ADD,               // a: xyzz, b: xyzz    -> xyzz
  C_NEG,               // a: xyzz             -> xyzz
  C_FROM_JAC,          // a: jac              -> xyzz
  C_TO_JAC_RAW,        // a: xyzz             -> jac
  C_TO_JAC_NORMALISED, // a: xyzz             -> jac
  C_MUL_U32,           // a: xyzz, aux: k     -> xyzz
  C_NOPS
};

template <class T>
__device__ T load_as(const uint8_t* base, size_t i) {
  return reinterpret_cast<const T*>(base)[i];
}

template <class C, int OP>
__global__ void curve_kernel(const uint8_t* a, const uint8_t* b, const uint32_t* aux, uint8_t* out, size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if constexpr (OP == C_TO_JAC_RAW || OP == C_TO_JAC_NORMALISED) {
    const xyzz_t p = load_as<xyzz_t>(a, i);
    reinterpret_cast<jac_t*>(out)[i] = OP == C_TO_JAC_RAW ? C::to_jac_raw(p) : C::to_jac_normalised(p);
    return;
  } else {
    xyzz_t r;
    if constexpr (OP == C_FROM_AFFINE) r = C::from_affine(load_as<affine_t>(a, i));
    else if constexpr (OP == C_DBL_AFFINE) {
      const affine_t p = load_as<affine_t>(a, i);
      r = C::dbl_affine(p.x, p.y);
    } else if constexpr (OP == C_FROM_JAC) r = C::from_jac(load_as<jac_t>(a, i));
    else {
      r = load_as<xyzz_t>(a, i);
      if constexpr (OP == C_MADD || OP == C_MADD_CALL) {
        const affine_t q = load_as<affine_t>(b, i);
        if (OP == C_MADD) C::madd(r, q.x, q.y);
        else C::madd_call(r, q.x, q.y);
      } else if constexpr (OP == C_MADD_SIGNED) C::madd_signed(r, load_as<affine_t>(b, i), aux[i] != 0);
      else if constexpr (OP == C_MADD_SIGNED_CALL) C::madd_signed_call(r, load_as<affine_t>(b, i), aux[i] != 0);
      else if constexpr (OP == C_DBL) r = C::dbl(r);
      else if constexpr (OP == C_ADD) C::add(r, load_as<xyzz_t>(b, i));
      else if constexpr (OP == C_NEG) r = C::neg(r);
      else if constexpr (OP == C_MUL_U32) r = C::mul_u32(r, aux[i]);
    }
    reinterpret_cast<xyzz_t*>(out)[i] = r;
  }
}

// ---- quad: four lanes per case ---------------------------------------------------------------------
// Quad q of the grid computes case q; its four lanes read the same operands, lane 0 writes the result.
template <class F, bool ADD>
__global__ void quad_kernel(const xyzz_t* acc, const xyzz_t* q, xyzz_t* out, size_t n) {
  const size_t c = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 2;
  if (c >= n) return;
  xyzz_t r = acc[c];
  if (ADD) Quad<F>::add(r, q[c]);
  else r = Quad<F>::dbl(r);
  if ((threadIdx.x & 3u) == 0) out[c] = r;
}

// every lane of the grid (a multiple of 32) holds in[lane] and writes what `down` returns to it
template <class F>
__global__ void quad_down_kernel(const xyzz_t* in, xyzz_t* out, int delta) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  out[i] = Quad<F>::down(in[i], delta);
}

// ---- plumbing ---------------------------------------------------------------------------------------
void check(cudaError_t e) {
  if (e != cudaSuccess) throw e;
}

// the multiplier reads M1..M3 from this translation unit's own copy of the constant array
void ensure_constants() {
  static bool done = false;
  if (!done) {
    check(upload_field_constants());
    done = true;
  }
}

// device buffers freed at scope exit
struct Dev {
  std::vector<void*> ptrs;
  ~Dev() {
    for (void* p : ptrs) cudaFree(p);
  }
  template <class T = uint8_t>
  T* alloc(size_t bytes) {
    void* p = nullptr;
    check(cudaMalloc(&p, bytes ? bytes : 16));
    ptrs.push_back(p);
    return reinterpret_cast<T*>(p);
  }
  template <class T = uint8_t>
  T* upload(const void* h, size_t bytes) {
    T* d = alloc<T>(bytes);
    if (bytes) check(cudaMemcpy(d, h, bytes, cudaMemcpyHostToDevice));
    return d;
  }
};

void download(void* h, const void* d, size_t bytes) {
  if (bytes) check(cudaMemcpy(h, d, bytes, cudaMemcpyDeviceToHost));
}

void finish_launch() {
  check(cudaGetLastError());
  check(cudaDeviceSynchronize());
}

template <class Body>
int guarded(Body body) {
  try {
    ensure_constants();
    body();
    return 0;
  } catch (cudaError_t e) {
    return (int)e;
  } catch (const std::exception&) {   // VDF_CUDA_CHECK inside CudaLaunch
    cudaError_t e = cudaGetLastError();
    return e != cudaSuccess ? (int)e : -1;
  }
}

unsigned blocks_of(size_t n, unsigned block) { return (unsigned)((n + block - 1) / block); }

template <class F, int OP>
void field_launch_op(int op, const fe* a, const fe* b, fe* o, uint8_t* fl, size_t n) {
  if constexpr (OP < F_NOPS) {
    if (op == OP) field_kernel<F, OP><<<blocks_of(n, 128), 128>>>(a, b, o, fl, n);
    else field_launch_op<F, OP + 1>(op, a, b, o, fl, n);
  } else {
    throw cudaErrorInvalidValue;
  }
}

template <class C, int OP>
void curve_launch_op(int op, const uint8_t* a, const uint8_t* b, const uint32_t* aux, uint8_t* o, size_t n) {
  if constexpr (OP < C_NOPS) {
    if (op == OP) curve_kernel<C, OP><<<blocks_of(n, 64), 64>>>(a, b, aux, o, n);
    else curve_launch_op<C, OP + 1>(op, a, b, aux, o, n);
  } else {
    throw cudaErrorInvalidValue;
  }
}

size_t curve_in_size(int op) {
  return op == C_FROM_AFFINE || op == C_DBL_AFFINE ? sizeof(affine_t) : op == C_FROM_JAC ? sizeof(jac_t) : sizeof(xyzz_t);
}
size_t curve_b_size(int op) {
  return op == C_ADD ? sizeof(xyzz_t)
         : (op == C_MADD || op == C_MADD_CALL || op == C_MADD_SIGNED || op == C_MADD_SIGNED_CALL) ? sizeof(affine_t)
                                                                                                     : 0;
}
size_t curve_out_size(int op) {
  return op == C_TO_JAC_RAW || op == C_TO_JAC_NORMALISED ? sizeof(jac_t) : sizeof(xyzz_t);
}

// AffineFwdFn -> BatchInvFn -> AffineBwdFn on one batch, as one round of msm_affine_rounds runs them
template <class F>
void affine_batch(const affine_t* aos, const fe* xs, const fe* ys, size_t npts, const uint32_t* ra, const uint32_t* rb,
                  uint32_t M, uint32_t T, uint32_t K, fe* hx, fe* hy) {
  Dev d;
  PointSrc in{nullptr, nullptr, nullptr};
  if (aos) in.aos = d.upload<affine_t>(aos, npts * sizeof(affine_t));
  else {
    in.xs = d.upload<fe>(xs, npts * sizeof(fe));
    in.ys = d.upload<fe>(ys, npts * sizeof(fe));
  }
  const uint32_t* dra = d.upload<uint32_t>(ra, M * sizeof(uint32_t));
  const uint32_t* drb = d.upload<uint32_t>(rb, M * sizeof(uint32_t));
  const uint32_t* dm = d.upload<uint32_t>(&M, sizeof(uint32_t));
  fe* prefix = d.alloc<fe>(M * sizeof(fe));
  fe* ptot = d.alloc<fe>(T * sizeof(fe));
  fe* ox = d.alloc<fe>(M * sizeof(fe));
  fe* oy = d.alloc<fe>(M * sizeof(fe));
  CudaLaunch L(0);
  L.run<128>(T, AffineFwdFn<F>{in, dra, drb, dm, T, K, prefix, ptot});
  L.run<64>((T + BatchInvFn<F>::J - 1) / BatchInvFn<F>::J, BatchInvFn<F>{ptot, T});
  L.run<128>(T, AffineBwdFn<F>{in, dra, drb, dm, T, K, prefix, ptot, ox, oy});
  check(cudaDeviceSynchronize());
  download(hx, ox, M * sizeof(fe));
  download(hy, oy, M * sizeof(fe));
}

template <class F>
void batch_inv(fe* hv, uint32_t n) {
  Dev d;
  fe* v = d.upload<fe>(hv, n * sizeof(fe));
  CudaLaunch L(0);
  L.run<64>((n + BatchInvFn<F>::J - 1) / BatchInvFn<F>::J, BatchInvFn<F>{v, n});
  check(cudaDeviceSynchronize());
  download(hv, v, n * sizeof(fe));
}

}  // namespace

extern "C" {
#pragma GCC visibility push(default)

// out: n field elements, or n bytes (0/1) for is_canonical / eq / is_zero.  b is read by the binary operations only
// but must hold n elements for every op.
int prims_field(int field, int op, const void* a, const void* b, void* out, size_t n) {
  return guarded([&] {
    Dev d;
    const fe* da = d.upload<fe>(a, n * sizeof(fe));
    const fe* db = d.upload<fe>(b, n * sizeof(fe));
    fe* o = d.alloc<fe>(n * sizeof(fe));
    uint8_t* fl = d.alloc(n);
    if (field == 0) field_launch_op<Fp, 0>(op, da, db, o, fl, n);
    else field_launch_op<Fq, 0>(op, da, db, o, fl, n);
    finish_launch();
    const bool flag = op == F_IS_CANONICAL || op == F_EQ || op == F_IS_ZERO;
    download(out, flag ? (const void*)fl : (const void*)o, flag ? n : n * sizeof(fe));
  });
}

// a: n inputs of the op's type (128-byte XYZZ, 64-byte affine or 96-byte Jacobian), b: the second operand where the op
// has one (else ignored), aux: n words (negate flag or k; ignored by the other ops, may be null)
int prims_curve(int curve, int op, const void* a, const void* b, const uint32_t* aux, void* out, size_t n) {
  return guarded([&] {
    if (op < 0 || op >= C_NOPS) throw cudaErrorInvalidValue;
    Dev d;
    const uint8_t* da = d.upload(a, n * curve_in_size(op));
    const uint8_t* db = curve_b_size(op) ? d.upload(b, n * curve_b_size(op)) : nullptr;
    const uint32_t* dx = (op == C_MADD_SIGNED || op == C_MADD_SIGNED_CALL || op == C_MUL_U32)
                             ? d.upload<uint32_t>(aux, n * sizeof(uint32_t)) : nullptr;
    uint8_t* o = d.alloc(n * curve_out_size(op));
    if (curve == 0) curve_launch_op<Pallas, 0>(op, da, db, dx, o, n);
    else curve_launch_op<Vesta, 0>(op, da, db, dx, o, n);
    finish_launch();
    download(out, o, n * curve_out_size(op));
  });
}

// op 0: out[c] = acc[c] + q[c] (Quad::add), op 1: out[c] = 2 acc[c] (Quad::dbl; q ignored).  Blocks of 64 lanes
// (16 quads, two warps); the grid is rounded up to whole warps.
int prims_quad(int curve, int op, const void* acc, const void* q, void* out, size_t n) {
  return guarded([&] {
    if (op != 0 && op != 1) throw cudaErrorInvalidValue;
    Dev d;
    const xyzz_t* da = d.upload<xyzz_t>(acc, n * sizeof(xyzz_t));
    const xyzz_t* dq = d.upload<xyzz_t>(q, n * sizeof(xyzz_t));
    xyzz_t* o = d.alloc<xyzz_t>(n * sizeof(xyzz_t));
    const unsigned blocks = blocks_of(4 * n, 64);
    if (curve == 0) {
      if (op == 0) quad_kernel<Fp, true><<<blocks, 64>>>(da, dq, o, n);
      else quad_kernel<Fp, false><<<blocks, 64>>>(da, dq, o, n);
    } else {
      if (op == 0) quad_kernel<Fq, true><<<blocks, 64>>>(da, dq, o, n);
      else quad_kernel<Fq, false><<<blocks, 64>>>(da, dq, o, n);
    }
    finish_launch();
    download(out, o, n * sizeof(xyzz_t));
  });
}

// out[lane] = Quad::down(in[lane], delta) over nlanes lanes (a multiple of 32), one warp per block
int prims_quad_down(int curve, const void* in, void* out, size_t nlanes, int delta) {
  return guarded([&] {
    if (nlanes % 32) throw cudaErrorInvalidValue;
    Dev d;
    const xyzz_t* di = d.upload<xyzz_t>(in, nlanes * sizeof(xyzz_t));
    xyzz_t* o = d.alloc<xyzz_t>(nlanes * sizeof(xyzz_t));
    if (curve == 0) quad_down_kernel<Fp><<<(unsigned)(nlanes / 32), 32>>>(di, o, delta);
    else quad_down_kernel<Fq><<<(unsigned)(nlanes / 32), 32>>>(di, o, delta);
    finish_launch();
    download(out, o, nlanes * sizeof(xyzz_t));
  });
}

// One batched-affine round over caller-built pair lists: output o = point ra[o] + point rb[o] (rb[o] = 0xffffffff:
// point ra[o] passes through).  aos != null: packed affine points read through the gather path, bit 31 of a
// reference negates; else SoA arrays xs / ys indexed by the reference.  Thread t of T owns outputs t, t + T, ...,
// at most K of them (M <= T * K).  out_x / out_y: M raw x and y coordinates, (0, 0) for the identity.
int prims_affine_batch(int curve, const void* aos, const void* xs, const void* ys, size_t npts, const uint32_t* ra,
                       const uint32_t* rb, uint32_t M, uint32_t T, uint32_t K, void* out_x, void* out_y) {
  return guarded([&] {
    if ((uint64_t)T * K < M || T == 0) throw cudaErrorInvalidValue;
    const affine_t* a = reinterpret_cast<const affine_t*>(aos);
    const fe *x = reinterpret_cast<const fe*>(xs), *y = reinterpret_cast<const fe*>(ys);
    fe *ox = reinterpret_cast<fe*>(out_x), *oy = reinterpret_cast<fe*>(out_y);
    if (curve == 0) affine_batch<Fp>(a, x, y, npts, ra, rb, M, T, K, ox, oy);
    else affine_batch<Fq>(a, x, y, npts, ra, rb, M, T, K, ox, oy);
  });
}

// v[i] <- 1 / v[i] in place (BatchInvFn, J elements per thread); no element may be zero
int prims_batch_inv(int field, void* v, uint32_t n) {
  return guarded([&] {
    if (field == 0) batch_inv<Fp>(reinterpret_cast<fe*>(v), n);
    else batch_inv<Fq>(reinterpret_cast<fe*>(v), n);
  });
}

#pragma GCC visibility pop
}  // extern "C"
