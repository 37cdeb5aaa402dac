// Library context shared by the C-ABI translation units (api_*.cu).  One process drives one GPU.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdio>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/vdfgpu.h"
#include "launch.cuh"
#include "msm.cuh"

namespace vdf {

struct ArgError : std::runtime_error {
  using std::runtime_error::runtime_error;
};
struct StateError : std::runtime_error {
  using std::runtime_error::runtime_error;
};

// Preallocated MSM workspace of one stream (see Arena in launch.cuh).  Grown on demand, never shrunk until
// vdfgpu_trim() / vdfgpu_shutdown().
struct Workspace {
  cudaStream_t stream = nullptr;
  Arena arena;
  uint8_t* block = nullptr;
  size_t block_bytes = 0;
  uint64_t last_use = 0;
  // persistent staging of the host entry points on this stream (scalars in, point out): stable device pointers
  // from call to call, which is what lets a latency-regime MSM be replayed as a CUDA graph
  fe* stage_sc = nullptr;
  size_t stage_cap = 0;
  jac_t* stage_out = nullptr;
};

// A latency-regime MSM (Nova-size commitments: ~50 dependent launches of 5-40 us each) captured once as a CUDA graph
// and replayed while plan, pointers and workspace block stay the same: no per-kernel launch gaps, no host-side
// pipeline code on the replay path.
struct MsmGraph {
  uint64_t key_hash = 0;
  std::vector<uint64_t> key;     // plan words, pointers, stream
  const void* gens_pts = nullptr;
  const void* block = nullptr;
  cudaGraphExec_t exec = nullptr;
  size_t launches = 0;
  uint64_t last_use = 0;
};

// one in-flight host-scalar MSM of the asynchronous API (vdfgpu_msm_submit / vdfgpu_msm_wait): its own stream
// carries the upload, the kernels and the read-back, so two slots overlap copies AND kernels
struct AsyncSlot {
  cudaStream_t stream = nullptr;
  fe* d_scalars = nullptr;
  size_t cap = 0;
  jac_t* d_out = nullptr;
  cudaEvent_t done = nullptr;
  bool busy = false;
};
constexpr int VDF_ASYNC_SLOTS = 4;

// Generator sets kept resident behind the literal pasta-msm entry points mult_pippenger_{pallas,vesta}, which
// receive the (fixed) points with every call: see api_core.cu "drop-in cache".
struct DropinEntry {
  int curve = 0;
  const void* host_ptr = nullptr;
  size_t n = 0;
  std::vector<size_t> sample_idx;       // ascending point indices whose bytes are kept below
  std::vector<uint8_t> sample_bytes;    // 65 bytes per sampled point (x, y, infinity flag; padding excluded)
  uint64_t full_hash = 0;               // VDFGPU_DROPIN_VERIFY=full
  vdfgpu_gens* gens = nullptr;
  uint64_t last_use = 0;
};

// Upload of PAGEABLE host memory (what a Rust Vec is) through pinned staging buffers filled by several host threads:
// the driver's own pageable path stages with one thread (~11 GB/s measured: 12 ms for the 128 MiB of 2^22 scalars).
struct UploadStage {
  static constexpr int THREADS = 6, SLOTS = 2;
  static constexpr size_t CHUNK = (size_t)4 << 20;
  uint8_t* pinned[THREADS][SLOTS] = {};
  cudaEvent_t ev[THREADS][SLOTS] = {};
  bool used[THREADS][SLOTS] = {};
  bool ready = false;
};

struct Context {
  std::mutex mu;          // guards this struct while work is ENQUEUED; released before a call blocks on the GPU
  bool ready = false;
  int device = -1;
  cudaStream_t own_stream = nullptr;        // library stream: used by every thread that has not set its own
  cudaStream_t copy_stream = nullptr;       // H2D of scalar chunks, overlapped with compute (vdfgpu_msm)
  cudaEvent_t chunk_ev[8] = {};             // chunk k of the scalars has arrived
  cudaEvent_t start_ev = nullptr;
  AsyncSlot slots[VDF_ASYNC_SLOTS];
  std::atomic<uint64_t> launches{0};
  StageProfile prof;      // stage timing of the most recent MSM (vdfgpu_profile_*)
  std::vector<std::unique_ptr<Workspace>> workspaces;
  std::vector<MsmGraph> graphs;
  uint64_t graph_replays = 0, graph_captures = 0;
  UploadStage upload;
  std::vector<DropinEntry> dropin;
  uint64_t dropin_hits = 0, dropin_misses = 0;
  uint64_t tick = 0;
};

Context& ctx();
void set_error(const std::string& msg);
void upload_constants_r1cs();   // api_r1cs.cu's copy of the constant-memory tables
void upload_constants_sumcheck();   // api_sumcheck.cu's
void require_ready();           // binds the calling thread to the library's device (lazy vdfgpu_init(0))

// The stream a call enqueues on: the calling THREAD's stream (vdfgpu_set_stream is per thread) or the library's.
cudaStream_t cur_stream();
// Ends a blocking entry point: records an event behind the work just enqueued; guarded() waits for it AFTER
// the context mutex is released, so other threads can enqueue meanwhile.
void sync_after_unlock(cudaStream_t s);
void wait_pending_sync();
void discard_pending_sync();   // a failed call leaves nothing behind for the next one on this thread
struct DeviceScope {   // restores the caller's current device on exit (the library binds its own for the call)
  int prev = -1;
  DeviceScope() { if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; cudaGetLastError(); } }
  ~DeviceScope() {
    int cur = -1;
    if (prev >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != prev) cudaSetDevice(prev);
  }
};

// RAII device buffer on the context stream (stream-ordered)
template <class T>
struct DevBuf {
  T* p = nullptr;
  cudaStream_t s = nullptr;
  DevBuf() = default;
  DevBuf(size_t count, cudaStream_t st) : s(st) {
    void* q = nullptr;
    VDF_CUDA_CHECK(cudaMallocAsync(&q, count * sizeof(T) + 16, st));
    p = reinterpret_cast<T*>(q);
  }
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), s(o.s) { o.p = nullptr; }
  DevBuf& operator=(DevBuf&& o) noexcept {
    if (this != &o) {
      release();
      p = o.p; s = o.s; o.p = nullptr;
    }
    return *this;
  }
  void release() {
    if (p) cudaFreeAsync(p, s);
    p = nullptr;
  }
  ~DevBuf() { release(); }
};

inline void h2d(void* dst, const void* src, size_t bytes, cudaStream_t s) {
  if (bytes) VDF_CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, s));
}
// h2d for scalar vectors coming from the caller: large pageable sources go through UploadStage
void h2d_scalars(void* dst, const void* src, size_t bytes, cudaStream_t s);
inline void d2h(void* dst, const void* src, size_t bytes, cudaStream_t s) {
  if (bytes) VDF_CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, s));
}
inline void d2d(void* dst, const void* src, size_t bytes, cudaStream_t s) {
  if (bytes) VDF_CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, s));
}

// The launch policy of the entry points: every kernel it launches counts in vdfgpu_launch_count().
inline CudaLaunch api_launch(cudaStream_t s, StageProfile* p = nullptr, Arena* a = nullptr) {
  return CudaLaunch(s, p, a, &ctx().launches);
}

// The ABI's field and curve ids as types: `body` (a generic lambda) is called with Fp{} or Fq{}, or with the curve,
// its coordinate field and its scalar field.  Any other id is an argument error "<who>: unknown field / curve".
template <class Body>
decltype(auto) with_field(int field, const char* who, Body&& body) {
  if (field == VDFGPU_FP) return body(Fp{});
  if (field == VDFGPU_FQ) return body(Fq{});
  throw ArgError(std::string(who) + ": unknown field");
}
template <class Body>
decltype(auto) with_curve(int curve, const char* who, Body&& body) {
  if (curve == VDFGPU_PALLAS) return body(Pallas{}, Fp{}, Fq{});
  if (curve == VDFGPU_VESTA) return body(Vesta{}, Fq{}, Fp{});
  throw ArgError(std::string(who) + ": unknown curve");
}

// wraps a C-ABI body: locks while the body enqueues, waits for the GPU outside the lock, maps exceptions to
// status codes + thread-local message, leaves the caller's current device as it found it
template <class Body>
int guarded(Body body) {
  DeviceScope dev;
  try {
    {
      std::lock_guard<std::mutex> lk(ctx().mu);
      body();
    }
    wait_pending_sync();
    return VDFGPU_OK;
  } catch (const ArgError& e) {
    discard_pending_sync();
    set_error(e.what());
    return VDFGPU_ERR_ARG;
  } catch (const StateError& e) {
    discard_pending_sync();
    set_error(e.what());
    return VDFGPU_ERR_STATE;
  } catch (const std::exception& e) {
    discard_pending_sync();
    set_error(e.what());
    return VDFGPU_ERR_CUDA;
  }
}

}  // namespace vdf

// handles ------------------------------------------------------------------------------------------
struct vdfgpu_gens {
  int curve = 0;
  size_t n = 0;            // points per level
  uint32_t flags = 0;
  uint32_t c = 0;          // window bits of the table (table mode)
  uint32_t W = 0;          // levels stored (1 in plain mode)
  vdf::affine_t* pts = nullptr;  // [W][n]
  int refs = 0;            // running instances and IPA calls in progress holding this set (vdfgpu_gens_destroy refuses
                           // while > 0)
};

// internal cross-TU entry: MSM over device scalars into a device point, on the calling thread's stream
namespace vdf {
// raw = true: the result is written as an un-normalised Jacobian point whatever the set's flags say (the host entry
// points then normalise it on the host, see normalise_after_sync).  replay = false: never run as a cached graph -- for
// points in a transient buffer, whose address keys a graph nothing will replay, and which would evict useful ones
void msm_on_device(vdfgpu_gens* g, size_t first, const fe* d_scalars, size_t n, jac_t* d_out, bool is_mont,
                   cudaStream_t stream = nullptr, bool raw = false, bool replay = true);
void msm_batch_on_device(vdfgpu_gens* g, const fe* const* d_scalars, const size_t* lens, uint32_t k, jac_t* d_out,
                         bool raw = false, bool replay = true);
// Host entry points that return a point to HOST memory let the device write the un-normalised Jacobian result and
// divide by Z on the host once the copy has landed: one field inversion is a strictly sequential chain of ~335
// multiplications -- 0.12 ms in a single GPU thread, ~15 us on a CPU core -- and the bytes are identical.  (Same
// split as the north star's: what cannot be parallelised stays on the host; Rust's to_affine() does this inversion on
// the host for pasta-msm's results today.)  `count` consecutive 96-byte points at host_ptr, after the pending wait.
void normalise_after_sync(void* host_ptr, size_t count, int curve);
// after the pending wait, before the normalisations: memcpy(dst, src, bytes) -- results land in a pinned bounce buffer
// with ONE asynchronous copy and are handed to the caller's (usually pageable) pointers on the host
void copy_after_sync(void* dst, const void* src, size_t bytes);
bool host_normalise_wanted(const vdfgpu_gens* g);
// a^-1 in Montgomery form, computed on the host (a != 0): the per-round challenge inverse of the IPA
fe host_inv(Fp, const fe& a);
fe host_inv(Fq, const fe& a);

// api_sumcheck.cu's building blocks, for the Spartan prover of the running instance (api_r1cs.cu).  Instances: Fp and
// Fq, K = 2 and 3.
template <int K>
struct MultiDot;
// eq(r) over 2^ell entries from ell challenges on the device
template <class F>
void eq_evals_enqueue(CudaLaunch& L, const fe* r_dev, size_t ell, fe* out_dev);
// K inner products over n entries into out[0, K) (sumcheck.cuh MultiDot); partial: sc_grid(n) K elements
template <class F, int K>
void multi_dot_enqueue(cudaStream_t st, const MultiDot<K>& d, size_t n, fe* partial, fe* out);
// per-thread pinned landing zone of small read-backs: 24 elements
fe* pinned_evals();
// the round loops of vdfgpu_sumcheck_{cubic,quad}[_dev] and vdfgpu_ipa_prove[_dev]: each is a whole call of its own
// (several guarded() sections, the callback between them), so it is called outside any guarded() section
int sumcheck(int field, const void* const* tables, int n_polys, bool on_host, size_t ell, vdfgpu_round_fn fn,
             void* user, void* final_host);
int ipa_prove(vdfgpu_gens* g, void* a_in, void* b_in, bool on_host, size_t ell, const void* u_scale_host,
              vdfgpu_ipa_round_fn fn, void* user, void* a_hat_host);

// a challenge the round loop can use: canonical (< m, so r = m is not a disguised 0) and not 0, which has no inverse
template <class F>
bool usable_challenge(const fe& r) {
  return F::is_canonical(r) && !F::is_zero(r);
}

// v[i] <- v[i]^-1 for non-zero v with ONE inversion (Montgomery's trick)
template <class F>
void batch_invert(std::vector<fe>& v) {
  if (v.empty()) return;
  std::vector<fe> pre(v.size());
  fe acc = F::one();
  for (size_t i = 0; i < v.size(); i++) {
    pre[i] = acc;
    acc = F::mul(acc, v[i]);
  }
  fe inv = host_inv(F{}, acc);
  for (size_t i = v.size(); i-- > 0;) {
    const fe vi = v[i];
    v[i] = F::mul(inv, pre[i]);
    inv = F::mul(inv, vi);
  }
}

// Batch verification of inner-product arguments (vdfgpu_ipa_verify_batch; notation in sumcheck.cuh), shared with the
// Spartan verifier (api_r1cs.cu).  Proof q's commitment is a short sum of terms, comm_a = sum_t coef[q][t] P[q][t]:
// vdfgpu_ipa_verify_batch has one term with coefficient 1, the Spartan opening comm_E + rho comm_W two.  Point j of
// proof q's commitment is at comm + 96 (q comm_stride + j), L_j at L + 96 (q lr_stride + j), R_j likewise.
struct IpaVerifyArgs {
  const uint8_t* comm; const uint8_t* L; const uint8_t* R;   // 96-byte Jacobian points
  const fe* r; const fe* a_hat; const fe* c; const fe* b_hat; const fe* u_scale; const fe* w;
  size_t terms = 1, comm_stride = 1, lr_stride = 0;
  const fe* coef = nullptr;          // [k][terms]; nullptr: every coefficient is 1
  const uint8_t* admit = nullptr;    // [k]: 0 for a proof the caller has already rejected; nullptr: all admitted
};
// Runs after the host checks inside the call's first guarded() section, on its stream, before the batch is enqueued:
// it may enqueue work and read-backs for the active proofs (ascending), which land behind the batch's one wait.
using IpaVerifyHook = void (*)(void* user, const std::vector<size_t>& active, cudaStream_t st);
// ok: k verdicts (zeroed first; fail closed).  `who` names the entry point in argument errors.
int ipa_verify_batch(vdfgpu_gens* g, size_t ell, size_t k, const IpaVerifyArgs& a, uint8_t* ok, const char* who,
                     IpaVerifyHook hook = nullptr, void* hook_user = nullptr);
}
