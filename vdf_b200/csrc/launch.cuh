// Launch policies.  Every kernel in this library is a functor `f(size_t i)` run over a 1-D index
// space; the pipelines (msm.cuh, r1cs.cuh, minroot.cuh) are templates over a policy L:
//
//   CudaLaunch  -- the product: real kernels on a CUDA stream, stream-ordered allocations.
//   HostLaunch  -- tests/emul only: the SAME functors executed by a CPU loop so the pipeline logic
//                  (digit recoding, counting sort, segmented bucket accumulation, reduction tree) can
//                  be checked against the oracle in a container without a GPU.  Never linked into
//                  libvdfgpu.so.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <map>
#include <stdexcept>
#include <string>

#include "field.cuh"

namespace vdf {

// ---- atomics usable from both policies ---------------------------------------------------------
VDF_HD uint32_t atomic_add_u32(uint32_t* p, uint32_t v) {
#if defined(__CUDA_ARCH__)
  return atomicAdd(p, v);
#else
  uint32_t old = *p;
  *p = old + v;
  return old;
#endif
}

VDF_HD uint32_t atomic_min_u32(uint32_t* p, uint32_t v) {
#if defined(__CUDA_ARCH__)
  return atomicMin(p, v);
#else
  uint32_t old = *p;
  if (v < old) *p = v;
  return old;
#endif
}

// ---- workspace arena ------------------------------------------------------------------------------
// Host-side bookkeeping of ONE preallocated device block per stream: the pipelines allocate and free their
// temporaries here (first fit, lowest address, 256-byte granules) instead of calling cudaMallocAsync /
// cudaFreeAsync ~30 times per MSM.  All users of one arena run on one stream, so a freed range may be handed
// out again at once (stream order protects it).  The same allocator run without a device block
// (PlanLaunch below) replays a pipeline's alloc/free sequence and yields its exact high-water mark, which is
// how the block is sized before the first launch.  Pointers are stable across calls of the same plan --
// the precondition for replaying a call as a CUDA graph.
class Arena {
 public:
  static constexpr size_t GRAN = 256;
  static constexpr size_t UNBOUNDED = (size_t)1 << 60;
  uint8_t* base = nullptr;   // device block; in measuring mode a fake non-null base that is never dereferenced
  size_t cap = 0;
  size_t high = 0;           // high-water mark since reset()

  void reset(size_t capacity) {
    free_.clear();
    live_.clear();
    free_[0] = capacity;
    cap = capacity;
    high = 0;
  }
  void* alloc(size_t bytes) {
    const size_t need = (bytes + GRAN - 1) / GRAN * GRAN + GRAN;   // one spare granule: kernels may over-read 16 B
    for (auto it = free_.begin(); it != free_.end(); ++it) {
      if (it->second < need) continue;
      const size_t off = it->first, rest = it->second - need;
      free_.erase(it);
      if (rest) free_[off + need] = rest;
      live_[off] = need;
      if (off + need > high) high = off + need;
      return base + off;
    }
    throw std::runtime_error("workspace arena exhausted (sizing pass and run disagree)");
  }
  void free(void* p) {
    if (!p) return;
    const size_t off = (size_t)(reinterpret_cast<uint8_t*>(p) - base);
    auto lv = live_.find(off);
    if (lv == live_.end()) throw std::runtime_error("workspace arena: free of an unknown block");
    size_t size = lv->second, start = off;
    live_.erase(lv);
    auto nx = free_.lower_bound(start);
    if (nx != free_.end() && nx->first == start + size) {   // merge with the block on the right
      size += nx->second;
      nx = free_.erase(nx);
    }
    if (nx != free_.begin()) {                              // ... and on the left
      auto pv = std::prev(nx);
      if (pv->first + pv->second == start) {
        pv->second += size;
        return;
      }
    }
    free_[start] = size;
  }

 private:
  std::map<size_t, size_t> free_, live_;   // offset -> size
};

// Sizing pass: the pipeline's host logic with no launches; afterwards arena.high is the workspace it needs.
// launches of one exclusive scan: short counter arrays (every latency-regime MSM) are scanned by ONE block
constexpr size_t SCAN_ONE_BLOCK_MAX = 8192;   // one chunk of the block; measured: 8.7 -> 5.0 us at 4096 counters, but 15 -> 52 us at 65536
static inline size_t scan_launches(size_t n) { return n <= SCAN_ONE_BLOCK_MAX ? 1 : 3; }

struct PlanLaunch {
  Arena arena;
  size_t launches = 0;
  PlanLaunch() {
    arena.base = reinterpret_cast<uint8_t*>((uintptr_t)1 << 40);
    arena.reset(Arena::UNBOUNDED);
  }
  void mark(int) {}
  template <class T>
  T* alloc(size_t count) { return reinterpret_cast<T*>(arena.alloc(count * sizeof(T))); }
  void free(void* p) { arena.free(p); }
  void zero(void*, size_t) {}
  void fill_ff(void*, size_t) {}
  template <int BLOCK = 256, int MINB = 1, class Fn>
  void run(size_t n, Fn) { if (n) launches++; }
  void exclusive_scan(const uint32_t*, uint32_t*, size_t n) {
    size_t tiles = (n + 2047) / 2048;
    if (tiles == 0) tiles = 1;
    uint32_t* t = alloc<uint32_t>(tiles);
    launches += scan_launches(n);
    free(t);
  }
};

#if defined(__CUDACC__)

#define VDF_CUDA_CHECK(expr)                                                                      \
  do {                                                                                            \
    cudaError_t e__ = (expr);                                                                     \
    if (e__ != cudaSuccess)                                                                       \
      throw std::runtime_error(std::string(#expr) + ": " + cudaGetErrorString(e__));              \
  } while (0)

// MINB = minimum resident blocks per SM the register allocation must allow (occupancy knob per kernel)
template <int BLOCK, int MINB, class Fn>
__global__ void __launch_bounds__(BLOCK, MINB) functor_kernel(Fn f, size_t n) {
  size_t i = (size_t)blockIdx.x * BLOCK + threadIdx.x;
  if (i < n) f(i);
}

// exclusive scan of u32 counters (3 phases); out has n+1 entries, out[n] = total
template <int BLOCK, int ITEMS>
__global__ void __launch_bounds__(BLOCK) scan_tile_kernel(const uint32_t* in, uint32_t* out, uint32_t* tile_sums,
                                                          size_t n) {
  __shared__ uint32_t warp_tot[BLOCK / 32];
  const size_t base = ((size_t)blockIdx.x * BLOCK + threadIdx.x) * ITEMS;
  uint32_t v[ITEMS];
  uint32_t sum = 0;
#pragma unroll
  for (int k = 0; k < ITEMS; k++) {
    v[k] = (base + k < n) ? in[base + k] : 0u;
    sum += v[k];
  }
  // warp inclusive scan of per-thread sums
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  uint32_t inc = sum;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += o;
  }
  if (lane == 31) warp_tot[wid] = inc;
  __syncthreads();
  if (wid == 0) {
    uint32_t w = (lane < BLOCK / 32) ? warp_tot[lane] : 0u;
    uint32_t winc = w;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      uint32_t o = __shfl_up_sync(0xffffffffu, winc, d);
      if (lane >= d) winc += o;
    }
    if (lane < BLOCK / 32) warp_tot[lane] = winc - w;  // exclusive warp offsets
    if (lane == 31) tile_sums[blockIdx.x] = winc;      // tile total (lanes >= BLOCK/32 add 0)
  }
  __syncthreads();
  uint32_t run = warp_tot[wid] + inc - sum;
#pragma unroll
  for (int k = 0; k < ITEMS; k++) {
    if (base + k < n) out[base + k] = run;
    run += v[k];
  }
}

// single block: exclusive scan of tile sums in place, total -> *total_out
template <int BLOCK>
__global__ void __launch_bounds__(BLOCK) scan_sums_kernel(uint32_t* tile_sums, size_t ntiles, uint32_t* total_out) {
  __shared__ uint32_t warp_tot[BLOCK / 32];
  __shared__ uint32_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (size_t base = 0; base < ntiles; base += BLOCK) {
    size_t i = base + threadIdx.x;
    uint32_t v = (i < ntiles) ? tile_sums[i] : 0u;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += o;
    }
    if (lane == 31) warp_tot[wid] = inc;
    __syncthreads();
    if (wid == 0) {
      uint32_t w = (lane < BLOCK / 32) ? warp_tot[lane] : 0u;
      uint32_t winc = w;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        uint32_t o = __shfl_up_sync(0xffffffffu, winc, d);
        if (lane >= d) winc += o;
      }
      if (lane < BLOCK / 32) warp_tot[lane] = winc - w;
    }
    __syncthreads();
    uint32_t excl = carry + warp_tot[wid] + inc - v;
    if (i < ntiles) tile_sums[i] = excl;
    __syncthreads();
    if (threadIdx.x == BLOCK - 1) carry = excl + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) *total_out = carry;
}

// the whole scan in ONE block for n <= SCAN_ONE_BLOCK_MAX (chunks of BLOCK * ITEMS counters with a running carry;
// out[n] = total): one launch of about 5 us instead of three dependent ones (about 9 us) in Nova-size commitments.
template <int BLOCK, int ITEMS>
__global__ void __launch_bounds__(BLOCK) scan_block_kernel(const uint32_t* in, uint32_t* out, size_t n) {
  __shared__ uint32_t warp_tot[BLOCK / 32];
  __shared__ uint32_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (size_t chunk = 0; chunk < n; chunk += (size_t)BLOCK * ITEMS) {
    const size_t base = chunk + (size_t)threadIdx.x * ITEMS;
    uint32_t v[ITEMS];
    uint32_t sum = 0;
#pragma unroll
    for (int k = 0; k < ITEMS; k++) {
      v[k] = (base + k < n) ? in[base + k] : 0u;
      sum += v[k];
    }
    uint32_t inc = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      uint32_t o = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += o;
    }
    if (lane == 31) warp_tot[wid] = inc;
    __syncthreads();
    if (wid == 0) {
      uint32_t w = (lane < BLOCK / 32) ? warp_tot[lane] : 0u;
      uint32_t winc = w;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        uint32_t o = __shfl_up_sync(0xffffffffu, winc, d);
        if (lane >= d) winc += o;
      }
      if (lane < BLOCK / 32) warp_tot[lane] = winc - w;
    }
    __syncthreads();
    uint32_t run = carry + warp_tot[wid] + inc - sum;
#pragma unroll
    for (int k = 0; k < ITEMS; k++) {
      if (base + k < n) out[base + k] = run;
      run += v[k];
    }
    __syncthreads();
    if (threadIdx.x == BLOCK - 1) carry = run;
    __syncthreads();
  }
  if (threadIdx.x == 0) out[n] = carry;
}

template <int BLOCK, int ITEMS>
__global__ void __launch_bounds__(BLOCK) scan_add_kernel(uint32_t* out, const uint32_t* tile_sums, size_t n) {
  const size_t base = ((size_t)blockIdx.x * BLOCK + threadIdx.x) * ITEMS;
  const uint32_t add = tile_sums[blockIdx.x];
#pragma unroll
  for (int k = 0; k < ITEMS; k++)
    if (base + k < n) out[base + k] += add;
}

// optional per-stage timing (bench.py's roofline leg): events recorded at stage boundaries
struct StageProfile {
  static constexpr int MAX_MARKS = 16;
  bool enabled = false;
  int n_marks = 0;
  int stage_of[MAX_MARKS];
  cudaEvent_t ev[MAX_MARKS];
  bool created = false;
};

struct CudaLaunch {
  cudaStream_t stream;
  size_t launches = 0;  // kernels launched through this policy (bench.py reports it)
  StageProfile* prof = nullptr;
  Arena* arena = nullptr;   // preallocated workspace of this stream; nullptr: stream-ordered pool allocations

  explicit CudaLaunch(cudaStream_t s, StageProfile* p = nullptr, Arena* a = nullptr) : stream(s), prof(p), arena(a) {}

  // stage boundary: everything enqueued until the next mark belongs to `stage`
  void mark(int stage) {
    if (!prof || !prof->enabled || prof->n_marks >= StageProfile::MAX_MARKS) return;
    if (!prof->created) {
      for (int i = 0; i < StageProfile::MAX_MARKS; i++) VDF_CUDA_CHECK(cudaEventCreate(&prof->ev[i]));
      prof->created = true;
    }
    prof->stage_of[prof->n_marks] = stage;
    VDF_CUDA_CHECK(cudaEventRecord(prof->ev[prof->n_marks], stream));
    prof->n_marks++;
  }

  template <class T>
  T* alloc(size_t count) {
    if (arena) return reinterpret_cast<T*>(arena->alloc(count * sizeof(T)));
    void* p = nullptr;
    VDF_CUDA_CHECK(cudaMallocAsync(&p, count * sizeof(T) + 16, stream));
    return reinterpret_cast<T*>(p);
  }
  void free(void* p) {
    if (!p) return;
    if (arena) arena->free(p);
    else VDF_CUDA_CHECK(cudaFreeAsync(p, stream));
  }
  void zero(void* p, size_t bytes) { VDF_CUDA_CHECK(cudaMemsetAsync(p, 0, bytes, stream)); }
  void fill_ff(void* p, size_t bytes) { VDF_CUDA_CHECK(cudaMemsetAsync(p, 0xff, bytes, stream)); }

  template <int BLOCK = 256, int MINB = 1, class Fn>
  void run(size_t n, Fn f) {
    if (n == 0) return;
    size_t blocks = (n + BLOCK - 1) / BLOCK;
    functor_kernel<BLOCK, MINB, Fn><<<(unsigned)blocks, BLOCK, 0, stream>>>(f, n);
    VDF_CUDA_CHECK(cudaGetLastError());
    launches++;
  }

  // out[0..n] = exclusive prefix sums of in[0..n), out[n] = total
  void exclusive_scan(const uint32_t* in, uint32_t* out, size_t n) {
    constexpr int BLOCK = 256, ITEMS = 8;
    size_t tiles = (n + (size_t)BLOCK * ITEMS - 1) / ((size_t)BLOCK * ITEMS);
    if (tiles == 0) tiles = 1;
    uint32_t* tile_sums = alloc<uint32_t>(tiles);   // (also in the one-block case: the sizing pass mirrors this)
    if (n <= SCAN_ONE_BLOCK_MAX) {
      scan_block_kernel<1024, 8><<<1, 1024, 0, stream>>>(in, out, n);
    } else {
      scan_tile_kernel<BLOCK, ITEMS><<<(unsigned)tiles, BLOCK, 0, stream>>>(in, out, tile_sums, n);
      scan_sums_kernel<256><<<1, 256, 0, stream>>>(tile_sums, tiles, out + n);
      scan_add_kernel<BLOCK, ITEMS><<<(unsigned)tiles, BLOCK, 0, stream>>>(out, tile_sums, n);
    }
    VDF_CUDA_CHECK(cudaGetLastError());
    launches += scan_launches(n);
    free(tile_sums);
  }
};

#endif  // __CUDACC__

// CPU loop policy: tests/emul only (see header comment)
struct HostLaunch {
  size_t launches = 0;
  void mark(int) {}
  template <class T>
  T* alloc(size_t count) {
    return reinterpret_cast<T*>(std::malloc(count * sizeof(T) + 16));
  }
  void free(void* p) { std::free(p); }
  void zero(void* p, size_t bytes) { std::memset(p, 0, bytes); }
  void fill_ff(void* p, size_t bytes) { std::memset(p, 0xff, bytes); }
  template <int BLOCK = 256, int MINB = 1, class Fn>
  void run(size_t n, Fn f) {
    for (size_t i = 0; i < n; i++) f(i);
    launches++;
  }
  void exclusive_scan(const uint32_t* in, uint32_t* out, size_t n) {
    uint32_t run = 0;
    for (size_t i = 0; i < n; i++) {
      uint32_t v = in[i];
      out[i] = run;
      run += v;
    }
    out[n] = run;
    launches += scan_launches(n);
  }
};

}  // namespace vdf
