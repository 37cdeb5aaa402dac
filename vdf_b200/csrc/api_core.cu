// C ABI, part 1: context, generator sets, MSM, batched MinRoot verification, measurement probes.
// See include/vdfgpu.h for the contract and the reference interfaces each entry point replaces.
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

#include "ctx.cuh"
#include "minroot.cuh"

namespace vdf {

static thread_local std::string g_error;
static thread_local cudaStream_t t_stream = nullptr;      // vdfgpu_set_stream: per calling thread
static thread_local cudaEvent_t t_sync_ev = nullptr;   // this thread's own "end of my call" event
static thread_local cudaEvent_t t_wait_ev = nullptr;   // what guarded() waits for after unlocking (or nullptr)

Context& ctx() {
  static Context c;
  return c;
}

void set_error(const std::string& msg) { g_error = msg; }

cudaStream_t cur_stream() { return t_stream ? t_stream : ctx().own_stream; }

void sync_after_unlock(cudaStream_t s) {
  if (!t_sync_ev) VDF_CUDA_CHECK(cudaEventCreateWithFlags(&t_sync_ev, cudaEventDisableTiming));
  VDF_CUDA_CHECK(cudaEventRecord(t_sync_ev, s));
  t_wait_ev = t_sync_ev;
}

static long env_long(const char* name, long dflt, long lo, long hi) {
  const char* s = std::getenv(name);
  if (!s || !*s) return dflt;
  long v = std::atol(s);
  return v < lo ? lo : (v > hi ? hi : v);
}

// ---- host-side normalisation of returned points (see ctx.cuh) ----------------------------------------------------
namespace hostfield {
typedef unsigned __int128 u128;
struct Mod { uint64_t m[4], one[4], inv; };   // modulus, R mod m, -m^-1 mod 2^64
static const Mod FP_MOD = {{0x992d30ed00000001ull, 0x224698fc094cf91bull, 0x0000000000000000ull, 0x4000000000000000ull},
                           {0x34786d38fffffffdull, 0x992c350be41914adull, 0xffffffffffffffffull, 0x3fffffffffffffffull},
                           0x992d30ecffffffffull};
static const Mod FQ_MOD = {{0x8c46eb2100000001ull, 0x224698fc0994a8ddull, 0x0000000000000000ull, 0x4000000000000000ull},
                           {0x5b2b3e9cfffffffdull, 0x992c350be3420567ull, 0xffffffffffffffffull, 0x3fffffffffffffffull},
                           0x8c46eb20ffffffffull};

static const Mod& mod_of(Fp) { return FP_MOD; }
static const Mod& mod_of(Fq) { return FQ_MOD; }
// the coordinate field of `curve`
static const Mod& coord_mod(int curve) {
  return with_curve(curve, "point_normalise_host", [](auto, auto f, auto) -> const Mod& { return mod_of(f); });
}

static void mul(uint64_t* r, const uint64_t* a, const uint64_t* b, const Mod& f) {   // Montgomery CIOS, 4 x 64
  uint64_t t[6] = {0, 0, 0, 0, 0, 0};
  for (int i = 0; i < 4; i++) {
    u128 c = 0;
    for (int j = 0; j < 4; j++) { c += (u128)a[j] * b[i] + t[j]; t[j] = (uint64_t)c; c >>= 64; }
    c += t[4]; t[4] = (uint64_t)c; t[5] = (uint64_t)(c >> 64);
    const uint64_t q = t[0] * f.inv;
    c = ((u128)q * f.m[0] + t[0]) >> 64;
    for (int j = 1; j < 4; j++) { c += (u128)q * f.m[j] + t[j]; t[j - 1] = (uint64_t)c; c >>= 64; }
    c += t[4]; t[3] = (uint64_t)c; t[4] = t[5] + (uint64_t)(c >> 64);
  }
  uint64_t s[4];
  u128 bw = 0;
  for (int j = 0; j < 4; j++) { u128 d = (u128)t[j] - f.m[j] - (uint64_t)bw; s[j] = (uint64_t)d; bw = (d >> 64) & 1; }
  const bool ge = t[4] != 0 || bw == 0;
  for (int j = 0; j < 4; j++) r[j] = ge ? s[j] : t[j];
}

static void inv(uint64_t* r, const uint64_t* a, const Mod& f) {   // a^(m-2)
  uint64_t e[4] = {f.m[0] - 2, f.m[1], f.m[2], f.m[3]};
  uint64_t acc[4];
  std::memcpy(acc, f.one, 32);
  for (int i = 255; i >= 0; i--) {
    mul(acc, acc, acc, f);
    if ((e[i >> 6] >> (i & 63)) & 1) mul(acc, acc, a, f);
  }
  std::memcpy(r, acc, 32);
}

// (X, Y, Z) Jacobian, Montgomery limbs -> (X / Z^2, Y / Z^3, 1), or all zero for the identity
static void normalise(uint8_t* p96, int curve) {
  const Mod& f = coord_mod(curve);
  uint64_t X[4], Y[4], Z[4];
  std::memcpy(X, p96, 32); std::memcpy(Y, p96 + 32, 32); std::memcpy(Z, p96 + 64, 32);
  if ((Z[0] | Z[1] | Z[2] | Z[3]) == 0) {
    std::memset(p96, 0, 96);
    return;
  }
  uint64_t zi[4], zi2[4], zi3[4];
  inv(zi, Z, f);
  mul(zi2, zi, zi, f);
  mul(zi3, zi2, zi, f);
  mul(X, X, zi2, f);
  mul(Y, Y, zi3, f);
  std::memcpy(p96, X, 32); std::memcpy(p96 + 32, Y, 32); std::memcpy(p96 + 64, f.one, 32);
}

// the same for m <= 16 points with one inversion: 1 / (Z_0 ... Z_{m-1}), then the individual inverses by back-substitution
static void normalise_batch(uint8_t* const* pts, size_t m, int curve) {
  const Mod& f = coord_mod(curve);
  uint64_t Z[16][4], pre[16][4], run[4];
  std::memcpy(run, f.one, 32);
  for (size_t k = 0; k < m; k++) {
    std::memcpy(Z[k], pts[k] + 64, 32);
    std::memcpy(pre[k], run, 32);
    if (Z[k][0] | Z[k][1] | Z[k][2] | Z[k][3]) mul(run, run, Z[k], f);
  }
  uint64_t inv_all[4];
  inv(inv_all, run, f);
  for (size_t k = m; k-- > 0;) {
    if ((Z[k][0] | Z[k][1] | Z[k][2] | Z[k][3]) == 0) {
      std::memset(pts[k], 0, 96);
      continue;
    }
    uint64_t zi[4], zi2[4], zi3[4], X[4], Y[4];
    mul(zi, inv_all, pre[k], f);
    mul(inv_all, inv_all, Z[k], f);
    std::memcpy(X, pts[k], 32); std::memcpy(Y, pts[k] + 32, 32);
    mul(zi2, zi, zi, f);
    mul(zi3, zi2, zi, f);
    mul(X, X, zi2, f);
    mul(Y, Y, zi3, f);
    std::memcpy(pts[k], X, 32); std::memcpy(pts[k] + 32, Y, 32); std::memcpy(pts[k] + 64, f.one, 32);
  }
}
}  // namespace hostfield

static fe host_inv_mod(const fe& a, const hostfield::Mod& f) {
  uint64_t x[4], r[4];
  std::memcpy(x, &a, 32);
  hostfield::inv(r, x, f);
  fe out;
  std::memcpy(&out, r, 32);
  return out;
}
fe host_inv(Fp, const fe& a) { return host_inv_mod(a, hostfield::FP_MOD); }
fe host_inv(Fq, const fe& a) { return host_inv_mod(a, hostfield::FQ_MOD); }

struct PendingNorm { void* p; size_t count; int curve; };
struct PendingCopy { void* dst; const void* src; size_t bytes; };
static thread_local std::vector<PendingNorm> t_norms;
static thread_local std::vector<PendingCopy> t_copies;

void copy_after_sync(void* dst, const void* src, size_t bytes) { t_copies.push_back({dst, src, bytes}); }

void normalise_after_sync(void* host_ptr, size_t count, int curve) { t_norms.push_back({host_ptr, count, curve}); }

bool host_normalise_wanted(const vdfgpu_gens* g) {
  return !(g->flags & VDFGPU_GENS_RAW_JACOBIAN) && env_long("VDFGPU_HOST_NORMALISE", 1, 0, 1) != 0;
}

void discard_pending_sync() {
  t_wait_ev = nullptr;
  t_norms.clear();
  t_copies.clear();
}

void wait_pending_sync() {
  cudaEvent_t ev = t_wait_ev;
  t_wait_ev = nullptr;
  std::vector<PendingNorm> norms;
  std::vector<PendingCopy> copies;
  norms.swap(t_norms);
  copies.swap(t_copies);
  if (ev) VDF_CUDA_CHECK(cudaEventSynchronize(ev));
  for (const PendingCopy& cp : copies) std::memcpy(cp.dst, cp.src, cp.bytes);
  // all points of one call share ONE inversion per curve (Montgomery's trick): a fold step returns two commitments
  for (int curve = 0; curve < 2; curve++) {
    uint8_t* pts[16];
    size_t m = 0;
    for (const PendingNorm& n : norms)
      for (size_t k = 0; k < n.count; k++) {
        if (n.curve != curve) continue;
        uint8_t* p = reinterpret_cast<uint8_t*>(n.p) + 96 * k;
        if (m < 16) pts[m++] = p;
        else hostfield::normalise(p, curve);
      }
    if (m == 1) hostfield::normalise(pts[0], curve);
    else if (m > 1) hostfield::normalise_batch(pts, m, curve);
  }
}


static void init_locked(int device) {
  Context& c = ctx();
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    throw std::runtime_error(std::string("no usable CUDA device (there is no CPU fallback): ") +
                             cudaGetErrorString(e));
  if (device < 0 || device >= count) throw ArgError("vdfgpu_init: device index out of range");
  if (c.ready && c.device == device) return;
  if (c.ready) throw StateError("vdfgpu_init: already bound to another device (one process per GPU)");
  VDF_CUDA_CHECK(cudaSetDevice(device));
  cudaDeviceProp prop;
  VDF_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10)
    throw std::runtime_error("vdfgpu: kernels are built for sm_100a only; found compute capability " +
                             std::to_string(prop.major) + "." + std::to_string(prop.minor));
  VDF_CUDA_CHECK(upload_field_constants());
  upload_constants_r1cs();
  upload_constants_sumcheck();
  VDF_CUDA_CHECK(cudaStreamCreateWithFlags(&c.own_stream, cudaStreamNonBlocking));
  VDF_CUDA_CHECK(cudaStreamCreateWithFlags(&c.copy_stream, cudaStreamNonBlocking));
  for (auto& e : c.chunk_ev) VDF_CUDA_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  VDF_CUDA_CHECK(cudaEventCreateWithFlags(&c.start_ev, cudaEventDisableTiming));
  // keep freed blocks in the stream-ordered pool (staging buffers of the host entry points)
  cudaMemPool_t pool;
  VDF_CUDA_CHECK(cudaDeviceGetDefaultMemPool(&pool, device));
  uint64_t threshold = UINT64_MAX;
  VDF_CUDA_CHECK(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold));
  c.device = device;
  c.ready = true;
}

void require_ready() {
  if (!ctx().ready) init_locked(0);
  int cur = -1;
  if (cudaGetDevice(&cur) != cudaSuccess || cur != ctx().device) VDF_CUDA_CHECK(cudaSetDevice(ctx().device));
}

// ---- pageable uploads -----------------------------------------------------------------------------------
void h2d_scalars(void* dst, const void* src, size_t bytes, cudaStream_t st) {
  if (!bytes) return;
  Context& c = ctx();
  UploadStage& u = c.upload;
  bool staged = bytes >= ((size_t)8 << 20) && env_long("VDFGPU_STAGED_UPLOAD", 1, 0, 1) != 0;
  if (staged) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, src) != cudaSuccess) {
      cudaGetLastError();
      staged = false;
    } else {
      staged = at.type == cudaMemoryTypeUnregistered;   // pinned / managed / device sources: plain asynchronous copy
    }
  }
  if (!staged) {
    VDF_CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
    return;
  }
  if (!u.ready) {
    for (int t = 0; t < UploadStage::THREADS; t++)
      for (int k = 0; k < UploadStage::SLOTS; k++) {
        VDF_CUDA_CHECK(cudaHostAlloc((void**)&u.pinned[t][k], UploadStage::CHUNK, cudaHostAllocDefault));
        VDF_CUDA_CHECK(cudaEventCreateWithFlags(&u.ev[t][k], cudaEventDisableTiming));
      }
    u.ready = true;
  }
  // copies run on the copy stream (the caller's stream may still be busy with the previous call's kernels, which
  // read the same staging destination: order the copy stream behind them first), and the caller's stream waits for
  // the last chunk
  VDF_CUDA_CHECK(cudaEventRecord(c.start_ev, st));
  VDF_CUDA_CHECK(cudaStreamWaitEvent(c.copy_stream, c.start_ev, 0));
  const size_t chunks = (bytes + UploadStage::CHUNK - 1) / UploadStage::CHUNK;
  const int device = c.device;
  std::string errors[UploadStage::THREADS];
  std::vector<std::thread> th;
  for (int t = 0; t < UploadStage::THREADS; t++)
    th.emplace_back([&, t] {
      try {
        VDF_CUDA_CHECK(cudaSetDevice(device));
        int slot = 0;
        for (size_t k = (size_t)t; k < chunks; k += UploadStage::THREADS, slot ^= 1) {
          const size_t off = k * UploadStage::CHUNK, len = off + UploadStage::CHUNK <= bytes ? UploadStage::CHUNK : bytes - off;
          if (u.used[t][slot]) VDF_CUDA_CHECK(cudaEventSynchronize(u.ev[t][slot]));   // its previous copy has drained
          std::memcpy(u.pinned[t][slot], reinterpret_cast<const uint8_t*>(src) + off, len);
          VDF_CUDA_CHECK(cudaMemcpyAsync(reinterpret_cast<uint8_t*>(dst) + off, u.pinned[t][slot], len, cudaMemcpyHostToDevice,
                                         c.copy_stream));
          VDF_CUDA_CHECK(cudaEventRecord(u.ev[t][slot], c.copy_stream));
          u.used[t][slot] = true;
        }
      } catch (const std::exception& e) {
        errors[t] = e.what();
      }
    });
  for (auto& x : th) x.join();
  for (auto& e : errors)
    if (!e.empty()) throw std::runtime_error("staged upload: " + e);
  VDF_CUDA_CHECK(cudaEventRecord(c.chunk_ev[0], c.copy_stream));
  VDF_CUDA_CHECK(cudaStreamWaitEvent(st, c.chunk_ev[0], 0));
}

// ---- workspaces --------------------------------------------------------------------------------------
static void graphs_drop_if(const void* block, const void* gens_pts) {
  Context& c = ctx();
  for (size_t i = 0; i < c.graphs.size();) {
    if ((block && c.graphs[i].block == block) || (gens_pts && c.graphs[i].gens_pts == gens_pts) || (!block && !gens_pts)) {
      cudaGraphExecDestroy(c.graphs[i].exec);
      c.graphs.erase(c.graphs.begin() + i);
    } else {
      i++;
    }
  }
}

static void workspace_release(Workspace& w) {
  if (w.block) {
    cudaStreamSynchronize(w.stream);
    graphs_drop_if(w.block, nullptr);
    cudaFree(w.block);
  }
  w.block = nullptr;
  w.block_bytes = 0;
}

static void workspace_release_all(Workspace& w) {
  workspace_release(w);
  if (w.stage_sc) cudaFree(w.stage_sc);
  if (w.stage_out) cudaFree(w.stage_out);
  w.stage_sc = nullptr;
  w.stage_out = nullptr;
  w.stage_cap = 0;
}

static void trim_locked() {
  Context& c = ctx();
  if (!c.ready) return;
  cudaDeviceSynchronize();
  graphs_drop_if(nullptr, nullptr);
  for (auto& w : c.workspaces) workspace_release_all(*w);
  c.workspaces.clear();
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, c.device) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
}

static bool workspaces_enabled() { return env_long("VDFGPU_WORKSPACE", 1, 0, 1) != 0; }

// the arena of `s`, holding at least `need` bytes, reset for a new call; nullptr when it cannot be had
// (then the caller falls back to stream-ordered pool allocations)
static Workspace* workspace_for(cudaStream_t s, size_t need, bool may_fail) {
  Context& c = ctx();
  Workspace* w = nullptr;
  for (auto& p : c.workspaces)
    if (p->stream == s) w = p.get();
  if (!w) {
    if (c.workspaces.size() >= 8) {   // evict the least recently used arena
      size_t lru = 0;
      for (size_t i = 1; i < c.workspaces.size(); i++)
        if (c.workspaces[i]->last_use < c.workspaces[lru]->last_use) lru = i;
      workspace_release_all(*c.workspaces[lru]);
      c.workspaces.erase(c.workspaces.begin() + lru);
    }
    c.workspaces.emplace_back(new Workspace());
    w = c.workspaces.back().get();
    w->stream = s;
  }
  w->last_use = ++c.tick;
  if (w->block_bytes < need) {
    workspace_release(*w);
    size_t want = need + need / 16;
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
      cudaGetLastError();
      want = need;
      e = cudaMalloc(&p, want);
    }
    if (e != cudaSuccess && !may_fail) {
      // last resort before failing the call: give back the other streams' idle arenas and the cached pool memory
      cudaGetLastError();
      for (auto& o : c.workspaces)
        if (o.get() != w) workspace_release(*o);
      cudaMemPool_t pool;
      if (cudaDeviceGetDefaultMemPool(&pool, c.device) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
      e = cudaMalloc(&p, want);
    }
    if (e != cudaSuccess) {
      cudaGetLastError();
      if (may_fail) return nullptr;
      throw std::runtime_error("msm workspace: cudaMalloc of " + std::to_string(need >> 20) + " MiB failed: " +
                               cudaGetErrorString(e));
    }
    w->block = reinterpret_cast<uint8_t*>(p);
    w->block_bytes = want;
  }
  w->arena.base = w->block;
  w->arena.reset(w->block_bytes);
  return w;
}

// persistent scalar / result staging of the host entry points on stream `s` (see Workspace)
static Workspace* staging_for(cudaStream_t s, size_t n) {
  Context& c = ctx();
  Workspace* w = nullptr;
  for (auto& p : c.workspaces)
    if (p->stream == s) w = p.get();
  if (!w) {
    w = workspace_for(s, 0, false);
  }
  if (!w->stage_out) VDF_CUDA_CHECK(cudaMalloc((void**)&w->stage_out, 4 * sizeof(jac_t)));
  if (w->stage_cap < n) {
    VDF_CUDA_CHECK(cudaStreamSynchronize(s));
    if (w->stage_sc) cudaFree(w->stage_sc);
    w->stage_sc = nullptr;
    w->stage_cap = 0;
    const size_t want = n + n / 8 + 64;
    cudaError_t e = cudaMalloc((void**)&w->stage_sc, want * sizeof(fe));
    if (e != cudaSuccess) {
      cudaGetLastError();
      VDF_CUDA_CHECK(cudaMalloc((void**)&w->stage_sc, (n + 1) * sizeof(fe)));
      w->stage_cap = n;
    } else {
      w->stage_cap = want;
    }
  }
  return w;
}

// ---- MSM dispatch -----------------------------------------------------------------------------------
static MsmPlan make_plan(const vdfgpu_gens* g, size_t n, bool is_mont, uint32_t batch = 1) {
  MsmPlan p;
  p.n = (uint32_t)n;
  p.batch = batch;
  for (uint32_t j = 0; j < MSM_MAX_BATCH; j++) p.len[j] = j < batch ? (uint32_t)n : 0u;
  p.table = (g->flags & VDFGPU_GENS_TABLE) ? 1u : 0u;
  p.c = p.table ? g->c : msm_pick_c(n, false);
  p.W = msm_windows(p.c);
  p.B = 1u << (p.c - 1);
  p.NB = p.table ? 1u : p.W;
  p.level_stride = g->n;
  p.is_mont = is_mont ? 1u : 0u;
  p.raw_jacobian = (g->flags & VDFGPU_GENS_RAW_JACOBIAN) ? 1u : 0u;
  // entries per accumulate thread: enough threads to fill 148 SMs, ranges long enough to amortise
  // the two boundary records each thread may emit
  size_t E = n * p.W * batch;
  size_t S = E / (148 * 768);
  // latency path: short serial chains per thread (measured on the Nova fold step, t = 1024: S = 16 -> 0.853 ms,
  // 8 -> 0.797, 4 -> 0.808: below 8 the extra boundary records cost more than the shorter chain saves)
  const size_t s_min = E <= (1u << 21) ? 8 : 32;
  if (S < s_min) S = s_min;
  if (S > 128) S = 128;
  p.S = (uint32_t)env_long("VDFGPU_MSM_S", (long)S, 1, 1 << 20);
  p.G = (uint32_t)env_long("VDFGPU_MSM_G", 16, 4, 1024);
  p.logm = (uint32_t)env_long("VDFGPU_MSM_LOGM", 3, 1, 8);
  p.rec_warp = (uint32_t)env_long("VDFGPU_MSM_RECWARP", 1, 0, 1);
  p.rec_bucket = (uint32_t)env_long("VDFGPU_MSM_RECBUCKET", 0, 0, 1);
  // batched-affine halving rounds (msm_affine.cuh): worth their fixed costs only in the throughput regime and
  // while the buckets still hold >= 12 entries on average
  p.affine_rounds = 0;
  if (E >= (1ull << 23)) {
    // measured on B200 (profiles/r1_experiments.md): -3 % at 2^20 points, -5 % at 2^22, -9 % at 2^24.  Halve while
    // a bucket keeps >= 12 entries on average and a round still has >= 4 M additions to pay for its fixed costs
    // (three small launches + one inversion latency); the XYZZ ranges finish the rest
    const size_t avg = E / ((size_t)p.NB * batch * p.B);
    while (p.affine_rounds < 5 && (avg >> (p.affine_rounds + 1)) >= 12 && (E >> (p.affine_rounds + 1)) >= (4u << 20))
      p.affine_rounds++;
  }
  p.affine_rounds = (uint32_t)env_long("VDFGPU_MSM_AFFINE", (long)p.affine_rounds, 0, 16);
  p.affine_K = (uint32_t)env_long("VDFGPU_MSM_AFFINE_K", 32, 1, 4096);
  if (E >= (1ull << 31)) p.affine_rounds = 0;   // 32-bit list positions, 0xffffffff reserved
  return p;
}

template <class C, class SF>
static size_t msm_workspace_bytes(const MsmPlan& p) {
  PlanLaunch PL;
  ScalarSet ss{{nullptr, nullptr, nullptr, nullptr}};
  msm_run<PlanLaunch, C, SF>(PL, p, nullptr, ss, nullptr);
  return PL.arena.high;
}

static size_t plan_bytes(int curve, const MsmPlan& p) {
  return with_curve(curve, "msm", [&](auto C, auto, auto SF) {
    return msm_workspace_bytes<decltype(C), decltype(SF)>(p);
  });
}

// Workspace for one MSM on stream `s`.  The affine rounds need ~52 B per sorted entry on top of the sort's 12 B:
// when that does not fit in what the device has left (2^26 points next to a 55 GB table and a second stream's
// arena), the plan drops them rather than failing.
static Workspace* plan_workspace(int curve, MsmPlan& p, cudaStream_t s) {
  if (!workspaces_enabled()) return nullptr;
  size_t need = plan_bytes(curve, p);
  Workspace* w = workspace_for(s, need, p.affine_rounds != 0);
  if (!w && p.affine_rounds) {
    p.affine_rounds = 0;
    need = plan_bytes(curve, p);
    w = workspace_for(s, need, false);
  }
  return w;
}

static void check_refs(const MsmPlan& p, const vdfgpu_gens* g, size_t n) {
  // point references are 31 bits (+ sign), sorted positions 32 bits
  if ((uint64_t)p.W * (p.table ? g->n : n) >= (1ull << 31))
    throw ArgError("msm: W * n exceeds the 31-bit point references (split the generator set, see vdfgpu.h)");
  if ((uint64_t)p.W * n * p.batch >= (1ull << 32)) throw ArgError("msm: too many sorted entries for one pass");
}

// ---- graph replay of latency-regime MSMs ------------------------------------------------------------------
static bool graphs_enabled() { return env_long("VDFGPU_GRAPH", 1, 0, 1) != 0; }
constexpr size_t GRAPH_MAX_ENTRIES = 1u << 22;   // sorted entries: above this the launch gaps no longer matter
constexpr size_t GRAPH_CACHE = 24;

static uint64_t mix64(uint64_t h, uint64_t v) {
  h ^= v + 0x9e3779b97f4a7c15ull + (h << 6) + (h >> 2);
  return h;
}

// runs `enqueue(L)` either directly or, for small plans on an arena, as a cached CUDA graph
template <class Enqueue>
static void msm_dispatch(vdfgpu_gens* g, const MsmPlan& p, Workspace* w, cudaStream_t st, const ScalarSet& ss,
                         const void* pts, const void* d_out, bool replay, Enqueue enqueue) {
  Context& c = ctx();
  const size_t E = (size_t)p.n * p.W * p.batch;
  if (!replay || !w || !graphs_enabled() || c.prof.enabled || E > GRAPH_MAX_ENTRIES) {
    CudaLaunch L = api_launch(st, &c.prof, w ? &w->arena : nullptr);
    enqueue(L);
    return;
  }
  std::vector<uint64_t> key = {(uint64_t)g->curve, p.n, p.c, p.W, p.B, p.NB, p.table, p.level_stride, p.S, p.G, p.logm, p.is_mont, p.batch,
                               p.len[0], p.len[1], p.len[2], p.len[3], p.raw_jacobian, p.rec_warp, p.rec_bucket, p.affine_rounds, p.affine_K};
  for (uint32_t j = 0; j < MSM_MAX_BATCH; j++) key.push_back((uint64_t)(uintptr_t)ss.v[j]);
  key.push_back((uint64_t)(uintptr_t)pts);
  key.push_back((uint64_t)(uintptr_t)d_out);
  key.push_back((uint64_t)(uintptr_t)w->block);
  key.push_back((uint64_t)(uintptr_t)st);
  uint64_t h = 0;
  for (uint64_t v : key) h = mix64(h, v);
  for (auto& e : c.graphs)
    if (e.key_hash == h && e.key == key) {
      e.last_use = ++c.tick;
      VDF_CUDA_CHECK(cudaGraphLaunch(e.exec, st));
      c.launches += e.launches;
      c.graph_replays++;
      return;
    }
  // capture (the arena is already large enough: nothing below allocates device memory); its launches count when
  // the graph runs
  cudaGraph_t graph = nullptr;
  CudaLaunch L(st, nullptr, &w->arena);
  VDF_CUDA_CHECK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
  try {
    enqueue(L);
  } catch (...) {
    cudaStreamEndCapture(st, &graph);
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    throw;
  }
  VDF_CUDA_CHECK(cudaStreamEndCapture(st, &graph));
  MsmGraph e;
  cudaError_t err = cudaGraphInstantiate(&e.exec, graph, 0);
  cudaGraphDestroy(graph);
  if (err != cudaSuccess) throw std::runtime_error(std::string("cudaGraphInstantiate: ") + cudaGetErrorString(err));
  e.key_hash = h;
  e.key = std::move(key);
  e.gens_pts = g->pts;
  e.block = w->block;
  e.launches = L.launches;
  e.last_use = ++c.tick;
  if (c.graphs.size() >= GRAPH_CACHE) {
    size_t lru = 0;
    for (size_t i = 1; i < c.graphs.size(); i++)
      if (c.graphs[i].last_use < c.graphs[lru].last_use) lru = i;
    cudaGraphExecDestroy(c.graphs[lru].exec);
    c.graphs.erase(c.graphs.begin() + lru);
  }
  VDF_CUDA_CHECK(cudaGraphLaunch(e.exec, st));
  c.launches += e.launches;
  c.graph_captures++;
  c.graphs.push_back(std::move(e));
}

void msm_on_device(vdfgpu_gens* g, size_t first, const fe* d_scalars, size_t n, jac_t* d_out, bool is_mont,
                   cudaStream_t stream, bool raw, bool replay) {
  if (first + n > g->n) throw ArgError("msm: more scalars than generators");
  Context& c = ctx();
  cudaStream_t st = stream ? stream : cur_stream();
  c.prof.n_marks = 0;
  MsmPlan p = make_plan(g, n, is_mont);
  if (raw) p.raw_jacobian = 1;
  check_refs(p, g, n);
  Workspace* w = n ? plan_workspace(g->curve, p, st) : nullptr;
  const affine_t* pts = g->pts + first;
  ScalarSet ss{{d_scalars, nullptr, nullptr, nullptr}};
  msm_dispatch(g, p, w, st, ss, pts, d_out, replay, [&](CudaLaunch& L) {
    with_curve(g->curve, "msm", [&](auto C, auto, auto SF) {
      msm_run<CudaLaunch, decltype(C), decltype(SF)>(L, p, pts, ss, d_out);
    });
  });
}

// Host-scalar MSM in point-range chunks: the H2D copy of chunk k+1 (copy stream) overlaps the digit / sort /
// accumulate stages of chunk k (compute stream); all chunks accumulate into ONE bucket array, so the bucket
// reduction and normalisation are paid once.  Result is identical to the single-pass MSM.
void msm_host_chunked(vdfgpu_gens* g, const void* h_scalars, size_t n, jac_t* d_out, fe* d_scalars, int chunks) {
  Context& c = ctx();
  cudaStream_t st = cur_stream();
  c.prof.n_marks = 0;
  CudaLaunch L = api_launch(st);
  MsmPlan full = make_plan(g, n, true);
  check_refs(full, g, n);
  const size_t NBK = (size_t)full.NB * full.B;
  DevBuf<xyzz_t> buckets(NBK, st), chunk_buckets(NBK, st);
  L.zero(buckets.p, NBK * sizeof(xyzz_t));
  // the copy stream must not run ahead of earlier work on the compute stream that may still read d_scalars
  VDF_CUDA_CHECK(cudaEventRecord(c.start_ev, st));
  VDF_CUDA_CHECK(cudaStreamWaitEvent(c.copy_stream, c.start_ev, 0));
  const size_t per = (n + chunks - 1) / chunks;
  for (int k = 0; k < chunks; k++) {
    size_t lo = (size_t)k * per, len = lo < n ? (lo + per <= n ? per : n - lo) : 0;
    if (len) VDF_CUDA_CHECK(cudaMemcpyAsync(d_scalars + lo, (const uint8_t*)h_scalars + lo * 32, len * 32,
                                            cudaMemcpyHostToDevice, c.copy_stream));
    VDF_CUDA_CHECK(cudaEventRecord(c.chunk_ev[k], c.copy_stream));
  }
  with_curve(g->curve, "msm", [&](auto C, auto, auto SF) {
    using Cv = decltype(C);
    for (int k = 0; k < chunks; k++) {
      size_t lo = (size_t)k * per, len = lo < n ? (lo + per <= n ? per : n - lo) : 0;
      VDF_CUDA_CHECK(cudaStreamWaitEvent(st, c.chunk_ev[k], 0));
      if (!len) continue;
      MsmPlan p = full;
      p.n = (uint32_t)len;
      p.len[0] = (uint32_t)len;
      ScalarSet ss{{d_scalars + lo, nullptr, nullptr, nullptr}};
      const affine_t* pts = g->pts + lo;
      xyzz_t* dst = k ? chunk_buckets.p : buckets.p;
      if (k) L.zero(dst, NBK * sizeof(xyzz_t));
      msm_accumulate<CudaLaunch, Cv, decltype(SF)>(L, p, pts, ss, dst);
      if (k) msm_merge_buckets<CudaLaunch, Cv>(L, full, buckets.p, chunk_buckets.p);
    }
    msm_finish<CudaLaunch, Cv>(L, full, buckets.p, d_out);
  });
}

// k scalar vectors over the same generators in ONE pass of the pipeline (one bucket set per vector):
// the latency of one MSM for k commitments.  d_out receives k points.
void msm_batch_on_device(vdfgpu_gens* g, const fe* const* d_scalars, const size_t* lens, uint32_t k, jac_t* d_out,
                         bool raw, bool replay) {
  if (k == 0 || k > MSM_MAX_BATCH) throw ArgError("msm_batch: batch size must be 1..4");
  size_t n = 0;
  for (uint32_t j = 0; j < k; j++) {
    if (lens[j] > g->n) throw ArgError("msm_batch: more scalars than generators");
    if (lens[j] > n) n = lens[j];
  }
  Context& c = ctx();
  cudaStream_t st = cur_stream();
  c.prof.n_marks = 0;
  MsmPlan p = make_plan(g, n, true, k);
  if (raw) p.raw_jacobian = 1;
  check_refs(p, g, n);
  ScalarSet ss{{nullptr, nullptr, nullptr, nullptr}};
  for (uint32_t j = 0; j < k; j++) {
    ss.v[j] = d_scalars[j];
    p.len[j] = (uint32_t)lens[j];
  }
  Workspace* w = n ? plan_workspace(g->curve, p, st) : nullptr;
  const affine_t* pts = g->pts;
  msm_dispatch(g, p, w, st, ss, pts, d_out, replay, [&](CudaLaunch& L) {
    with_curve(g->curve, "msm", [&](auto C, auto, auto SF) {
      msm_run<CudaLaunch, decltype(C), decltype(SF)>(L, p, pts, ss, d_out);
    });
  });
}

static void build_table(vdfgpu_gens* g, CudaLaunch& L) {
  // levels 1..W-1: level[l] = 2^c * level[l-1]
  for (uint32_t l = 1; l < g->W; l++) {
    const affine_t* prev = g->pts + (size_t)(l - 1) * g->n;
    affine_t* next = g->pts + (size_t)l * g->n;
    size_t threads = (g->n + 7) / 8;
    with_curve(g->curve, "gens", [&](auto C, auto BF, auto) {
      L.run<128>(threads, TableLevelFn<decltype(C), decltype(BF)>{prev, next, g->n, g->c});
    });
  }
}

// the arguments of a new generator set, checked before any device work
static void gens_check(int curve, size_t n, uint32_t window_bits) {
  with_curve(curve, "gens", [](auto, auto, auto) {});
  if (n == 0) throw ArgError("gens: empty generator set");
  if (window_bits != 0 && (window_bits < 2 || window_bits > 24)) throw ArgError("gens: window_bits out of range");
}

// the one release path of a generator set: failed creation, drop-in eviction, vdfgpu_gens_destroy
struct GensRelease {
  void operator()(vdfgpu_gens* g) const {
    graphs_drop_if(nullptr, g->pts);
    cudaFree(g->pts);
    delete g;
  }
};
using GensPtr = std::unique_ptr<vdfgpu_gens, GensRelease>;

static GensPtr gens_alloc(int curve, size_t n, uint32_t flags, uint32_t window_bits) {
  const bool table = flags & VDFGPU_GENS_TABLE;
  if (!window_bits) window_bits = (uint32_t)env_long("VDFGPU_WINDOW_BITS", 0, 0, 24);   // tuning knob; 0 = by size
  if (window_bits == 1) window_bits = 2;
  const uint32_t c = window_bits ? window_bits : msm_pick_c(n, table), W = table ? msm_windows(c) : 1;
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, (size_t)W * n * sizeof(affine_t));
  if (e != cudaSuccess) throw std::runtime_error(std::string("gens: cudaMalloc failed: ") + cudaGetErrorString(e));
  GensPtr g(new vdfgpu_gens());
  g->curve = curve;
  g->n = n;
  g->flags = flags;
  g->c = c;
  g->W = W;
  g->pts = reinterpret_cast<affine_t*>(p);
  return g;
}

// a resident set of the caller's 72-byte affine points (vdfgpu_gens_create, the drop-in cache)
static GensPtr gens_upload(int curve, const void* points72_host, size_t n, uint32_t flags, uint32_t window_bits,
                           cudaStream_t st) {
  GensPtr g = gens_alloc(curve, n, flags, window_bits);
  CudaLaunch L = api_launch(st);
  DevBuf<uint8_t> raw(n * 72, st);
  h2d(raw.p, points72_host, n * 72, st);
  L.run<256>(n, RepackFn{raw.p, g->pts});
  if (flags & VDFGPU_GENS_TABLE) build_table(g.get(), L);
  return g;
}

template <class F>
static void minroot_check_dispatch(CudaLaunch& L, const void* res, const void* orig, const uint64_t* t_each,
                                   uint64_t t_uniform, size_t n, uint8_t* ok) {
  // 32-thread blocks: 2^16 chains are only ~3.5 blocks of 128 per SM, and whole blocks cannot be split across
  // SMs (4 vs 3 resident blocks = 14 % imbalance); 2048 one-warp blocks spread evenly over the 148 SMs
  L.run<32>(n, MinRootCheckFn<F>{reinterpret_cast<const state_t*>(res), reinterpret_cast<const state_t*>(orig),
                                 t_each, t_uniform, ok});
}

template <class F>
struct FieldMulFn {
  const fe* a; const fe* b; fe* out; uint32_t iters;
  VDF_HD void operator()(size_t i) const {
    fe x = fe_load(a + i), y = fe_load(b + i);
    // bit 31 of iters selects the out-of-line multiplier (latency probe of the call overhead), bit 30 the
    // dedicated squaring (x <- x^2, b unused)
    const uint32_t n_it = iters & 0x3fffffffu;
    if (iters & 0x40000000u) {
#pragma unroll 1
      for (uint32_t k = 0; k < n_it; k++) x = F::sqr(x);
    } else if (iters >> 31) {
#if defined(__CUDA_ARCH__)
#pragma unroll 1
      for (uint32_t k = 0; k < n_it; k++) x = F::mul_call(x, y);
#endif
    } else {
#pragma unroll 1
      for (uint32_t k = 0; k < n_it; k++) x = F::mul(x, y);
    }
    fe_store(out + i, x);
  }
};

// ---- integer pipe probes --------------------------------------------------------------------------
// Register-only multiply-pipe probes.  Multiplicands are loop-variant (fed from the other accumulators)
// so nothing is hoisted: MODE 0 = 32x32+64 -> 64 multiply-adds in carry chains (IMAD.WIDE.U32[.X]),
// MODE 1 = low-half multiply-adds (IMAD), MODE 2 = add-with-carry chains (IADD3.X).
template <int MODE>
__global__ void __launch_bounds__(256) imad_probe_kernel(uint32_t* sink, uint32_t seed, int iters) {
  uint32_t x[16], y[8];
#pragma unroll
  for (int k = 0; k < 16; k++) x[k] = k * 0x9e3779b9u + seed + threadIdx.x;
#pragma unroll
  for (int k = 0; k < 8; k++) y[k] = (k ^ seed) * 2654435761u + blockIdx.x;
#pragma unroll 1
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int rep = 0; rep < 4; rep++) {
#pragma unroll
      for (int s = 0; s < 2; s++) {
        uint32_t* a = x + 8 * s;
        const uint32_t* m = y + 4 * s;
        if (MODE == 0) {
          asm volatile("mad.lo.cc.u32 %0, %8, %12, %0; madc.hi.cc.u32 %1, %8, %12, %1;"
                       "madc.lo.cc.u32 %2, %9, %12, %2; madc.hi.cc.u32 %3, %9, %12, %3;"
                       "madc.lo.cc.u32 %4, %10, %12, %4; madc.hi.cc.u32 %5, %10, %12, %5;"
                       "madc.lo.cc.u32 %6, %11, %12, %6; madc.hi.u32 %7, %11, %12, %7;"
                       : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7])
                       : "r"(m[0]), "r"(m[1]), "r"(m[2]), "r"(m[3]), "r"(x[(8 * s + 11 + rep) & 15]));
        } else if (MODE == 1) {
#pragma unroll
          for (int k = 0; k < 4; k++)
            asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+r"(a[k]) : "r"(m[k]), "r"(x[(8 * s + 11 + rep) & 15]));
        } else {
          asm volatile("add.cc.u32 %0, %0, %8; addc.cc.u32 %1, %1, %9; addc.cc.u32 %2, %2, %10; addc.cc.u32 %3, %3, %11;"
                       "addc.cc.u32 %4, %4, %8; addc.cc.u32 %5, %5, %9; addc.cc.u32 %6, %6, %10; addc.u32 %7, %7, %11;"
                       : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7])
                       : "r"(m[0]), "r"(m[1]), "r"(m[2]), "r"(m[3]));
        }
      }
    }
#pragma unroll
    for (int k = 0; k < 8; k++) y[k] ^= x[k + (k & 1) * 8];
  }
  uint32_t sacc = 0;
#pragma unroll
  for (int k = 0; k < 16; k++) sacc ^= x[k];
  if (sacc == 0x1234567u) sink[0] = sacc;
}

// operations of the probed kind per thread per loop iteration
template <int MODE>
static double probe_rate(cudaStream_t st, uint32_t* sink) {
  const int blocks = 148 * 8, iters = 2048;
  const double ops_per_iter = MODE == 2 ? 64.0 : 32.0;   // 4 reps x 2 sets x (4 products | 8 adds)
  cudaEvent_t e0, e1;
  VDF_CUDA_CHECK(cudaEventCreate(&e0));
  VDF_CUDA_CHECK(cudaEventCreate(&e1));
  for (int w = 0; w < 2; w++) imad_probe_kernel<MODE><<<blocks, 256, 0, st>>>(sink, 12345u, iters);
  VDF_CUDA_CHECK(cudaEventRecord(e0, st));
  imad_probe_kernel<MODE><<<blocks, 256, 0, st>>>(sink, 12345u, iters);
  VDF_CUDA_CHECK(cudaEventRecord(e1, st));
  VDF_CUDA_CHECK(cudaEventSynchronize(e1));
  float ms = 0;
  VDF_CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  double ops = (double)blocks * 256.0 * iters * ops_per_iter;
  return ops / (ms * 1e-3);
}

}  // namespace vdf

using namespace vdf;

extern "C" {
#pragma GCC visibility push(default)

int vdfgpu_init(int device) {
  return guarded([&] { init_locked(device); });
}

static void dropin_clear_locked();

int vdfgpu_shutdown(void) {
  return guarded([&] {
    Context& c = ctx();
    if (!c.ready) return;
    VDF_CUDA_CHECK(cudaSetDevice(c.device));
    cudaDeviceSynchronize();
    dropin_clear_locked();
    trim_locked();
    if (c.own_stream) cudaStreamDestroy(c.own_stream);
    if (c.copy_stream) cudaStreamDestroy(c.copy_stream);
    if (c.upload.ready) {
      for (int t = 0; t < UploadStage::THREADS; t++)
        for (int k = 0; k < UploadStage::SLOTS; k++) {
          cudaFreeHost(c.upload.pinned[t][k]);
          cudaEventDestroy(c.upload.ev[t][k]);
        }
      c.upload = UploadStage();
    }
    for (auto& e : c.chunk_ev) { if (e) cudaEventDestroy(e); e = nullptr; }
    if (c.start_ev) cudaEventDestroy(c.start_ev);
    c.start_ev = nullptr;
    for (auto& sl : c.slots) {
      if (sl.done) cudaEventDestroy(sl.done);
      if (sl.d_scalars) cudaFree(sl.d_scalars);
      if (sl.d_out) cudaFree(sl.d_out);
      if (sl.stream) cudaStreamDestroy(sl.stream);
      sl = AsyncSlot();
    }
    c.copy_stream = nullptr;
    c.own_stream = nullptr;
    t_stream = nullptr;
    c.ready = false;
    c.device = -1;
  });
}

int vdfgpu_trim(void) {
  return guarded([&] {
    for (auto& sl : ctx().slots)
      if (sl.busy) throw StateError("vdfgpu_trim: an asynchronous MSM is still in flight");
    if (ctx().ready) VDF_CUDA_CHECK(cudaSetDevice(ctx().device));
    trim_locked();
  });
}

int vdfgpu_device_count(void) {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess) return 0;
  return count;
}

const char* vdfgpu_last_error(void) { return g_error.c_str(); }

const char* vdfgpu_version(void) { return "vdfgpu 0.1 (sm_100a)"; }

int vdfgpu_set_stream(void* cuda_stream) {
  return guarded([&] {
    require_ready();
    t_stream = reinterpret_cast<cudaStream_t>(cuda_stream);   // nullptr: back to the library stream
  });
}

int vdfgpu_synchronize(void) {
  return guarded([&] {
    require_ready();
    sync_after_unlock(cur_stream());
  });
}

uint64_t vdfgpu_launch_count(void) { return ctx().launches.load(); }

int vdfgpu_profile_enable(int on) {
  return guarded([&] { ctx().prof.enabled = on != 0; });
}

int vdfgpu_profile_read(double* stage_ms, int n_stages) {
  return guarded([&] {
    require_ready();
    Context& c = ctx();
    if (!stage_ms || n_stages < 1) throw ArgError("profile_read: bad arguments");
    for (int i = 0; i < n_stages; i++) stage_ms[i] = 0.0;
    if (c.prof.n_marks < 2) throw StateError("profile_read: no profiled MSM (call vdfgpu_profile_enable(1) first)");
    VDF_CUDA_CHECK(cudaEventSynchronize(c.prof.ev[c.prof.n_marks - 1]));
    for (int k = 0; k + 1 < c.prof.n_marks; k++) {
      float ms = 0;
      VDF_CUDA_CHECK(cudaEventElapsedTime(&ms, c.prof.ev[k], c.prof.ev[k + 1]));
      int st = c.prof.stage_of[k];
      if (st >= 0 && st < n_stages) stage_ms[st] += ms;
    }
  });
}

// ---- generator sets ------------------------------------------------------------------------------------
int vdfgpu_gens_create(int curve, const void* points_affine72_host, size_t n, uint32_t flags,
                       uint32_t window_bits, vdfgpu_gens** out) {
  return guarded([&] {
    if (!out || !points_affine72_host) throw ArgError("gens_create: null pointer");
    gens_check(curve, n, window_bits);
    require_ready();
    GensPtr g = gens_upload(curve, points_affine72_host, n, flags, window_bits, cur_stream());
    sync_after_unlock(cur_stream());
    *out = g.release();
  });
}

int vdfgpu_gens_progression(int curve, const void* k0_le32, const void* d_le32, size_t n, uint32_t flags,
                            uint32_t window_bits, vdfgpu_gens** out) {
  return guarded([&] {
    if (!out || !k0_le32 || !d_le32) throw ArgError("gens_progression: null pointer");
    gens_check(curve, n, window_bits);
    const size_t threads = (n + PROG_CH - 1) / PROG_CH;
    if (threads >= (1ull << 32)) throw ArgError("gens_progression: n too large");
    require_ready();
    GensPtr g = gens_alloc(curve, n, flags, window_bits);
    CudaLaunch L = api_launch(cur_stream());
    fe k0, d;
    std::memcpy(k0.v, k0_le32, 32);
    std::memcpy(d.v, d_le32, 32);
    DevBuf<ProgSetup> setup(1, cur_stream());
    with_curve(curve, "gens", [&](auto C, auto BF, auto) {
      L.run<32>(1, ProgressionSetupFn<decltype(C), decltype(BF)>{k0, d, setup.p});
      L.run<128>(threads, ProgressionFn<decltype(C), decltype(BF)>{setup.p, g->pts, n});
    });
    if (flags & VDFGPU_GENS_TABLE) build_table(g.get(), L);
    sync_after_unlock(cur_stream());
    *out = g.release();
  });
}

int vdfgpu_gens_export(const vdfgpu_gens* g, size_t first, size_t count, void* points_affine72_host) {
  return guarded([&] {
    if (!g || !points_affine72_host) throw ArgError("gens_export: null pointer");
    if (first + count > (size_t)g->W * g->n) throw ArgError("gens_export: range out of bounds");
    require_ready();
    CudaLaunch L = api_launch(cur_stream());
    DevBuf<uint8_t> raw(count * 72, cur_stream());
    L.run<256>(count, UnpackFn{g->pts + first, raw.p});
    d2h(points_affine72_host, raw.p, count * 72, cur_stream());
    sync_after_unlock(cur_stream());
  });
}

size_t vdfgpu_gens_len(const vdfgpu_gens* g) { return g ? g->n : 0; }

uint32_t vdfgpu_gens_window_bits(const vdfgpu_gens* g, size_t n) {
  if (!g) return 0;
  return (g->flags & VDFGPU_GENS_TABLE) ? g->c : msm_pick_c(n, false);
}

uint32_t vdfgpu_gens_affine_rounds(const vdfgpu_gens* g, size_t n) {
  if (!g || n == 0 || n > g->n) return 0;
  return make_plan(g, n, true).affine_rounds;
}

int vdfgpu_gens_destroy(vdfgpu_gens* g) {
  return guarded([&] {
    if (!g) return;
    if (g->refs > 0)
      throw StateError("gens_destroy: a running instance or an inner-product argument in progress still uses this "
                       "generator set");
    if (ctx().ready) {
      VDF_CUDA_CHECK(cudaSetDevice(ctx().device));
      cudaDeviceSynchronize();   // MSMs on any stream (asynchronous slots, other threads) may still read the points
    }
    GensRelease()(g);
  });
}

// ---- MSM -------------------------------------------------------------------------------------------------
int vdfgpu_msm(vdfgpu_gens* g, const void* scalars32_host, size_t n, void* out_point96_host) {
  return guarded([&] {
    if (!g || !out_point96_host || (n && !scalars32_host)) throw ArgError("msm: null pointer");
    require_ready();
    Context& c = ctx();
    if (n > g->n) throw ArgError("msm: more scalars than generators");
    if (workspaces_enabled() && !std::getenv("VDFGPU_MSM_CHUNKS")) {
      // persistent staging buffers of this stream: stable pointers, so a Nova-size commitment replays as a graph
      cudaStream_t st = cur_stream();
      Workspace* ws = staging_for(st, n);
      h2d_scalars(ws->stage_sc, scalars32_host, n * 32, st);
      const bool hn = host_normalise_wanted(g);
      msm_on_device(g, 0, ws->stage_sc, n, ws->stage_out, true, nullptr, hn);
      d2h(out_point96_host, ws->stage_out, sizeof(jac_t), st);
      sync_after_unlock(st);
      if (hn) normalise_after_sync(out_point96_host, 1, g->curve);
      return;
    }
    DevBuf<fe> sc(n ? n : 1, cur_stream());
    DevBuf<jac_t> res(1, cur_stream());
    // Chunked schedule (H2D of chunk k+1 under the accumulation of chunk k): measured on B200 at n = 2^22 the
    // per-chunk fixed costs (sparser buckets, extra sort passes, bucket merge) cancel the ~1.2 ms of hidden
    // copy (14.1 ms with 1 or 2 chunks, 14.8 with 4), so the default stays one chunk; VDFGPU_MSM_CHUNKS overrides.
    int chunks = 1;
    if (const char* s = std::getenv("VDFGPU_MSM_CHUNKS")) chunks = std::atoi(s);
    if (chunks < 1) chunks = 1;
    if (chunks > 8) chunks = 8;
    if (chunks > 1 && n >= 1024) {
      msm_host_chunked(g, scalars32_host, n, res.p, sc.p, chunks);
    } else {
      h2d(sc.p, scalars32_host, n * 32, cur_stream());
      msm_on_device(g, 0, sc.p, n, res.p, true);
    }
    d2h(out_point96_host, res.p, sizeof(jac_t), cur_stream());
    sync_after_unlock(cur_stream());
  });
}

// Asynchronous host-scalar MSM.  Every slot owns a stream that carries its upload, kernels and read-back, so with
// two slots in flight the upload of one call AND its latency-bound stages (inversions, record levels, bucket
// reduction: ~2 ms of a 2^22-point MSM at < 10 % of the warp slots) run under the multiply-bound kernels of the
// other.  Each stream has its own workspace arena.
int vdfgpu_msm_submit(vdfgpu_gens* g, const void* scalars32_host, size_t n, void* out_point96_host, int slot) {
  return guarded([&] {
    if (!g || !out_point96_host || (n && !scalars32_host)) throw ArgError("msm_submit: null pointer");
    if (slot < 0 || slot >= VDF_ASYNC_SLOTS) throw ArgError("msm_submit: slot out of range");
    if (n > g->n) throw ArgError("msm_submit: more scalars than generators");
    require_ready();
    Context& c = ctx();
    AsyncSlot& s = c.slots[slot];
    if (s.busy) throw StateError("msm_submit: slot still in flight (call vdfgpu_msm_wait first)");
    if (!s.stream) {
      VDF_CUDA_CHECK(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
      VDF_CUDA_CHECK(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
      VDF_CUDA_CHECK(cudaMalloc((void**)&s.d_out, sizeof(jac_t)));
    }
    if (s.cap < n) {
      VDF_CUDA_CHECK(cudaStreamSynchronize(s.stream));
      if (s.d_scalars) VDF_CUDA_CHECK(cudaFree(s.d_scalars));
      s.d_scalars = nullptr;
      s.cap = 0;
      VDF_CUDA_CHECK(cudaMalloc((void**)&s.d_scalars, (n ? n : 1) * sizeof(fe)));
      s.cap = n;
    }
    // the generator set may have been built on the caller's stream just before: order the slot behind it
    VDF_CUDA_CHECK(cudaEventRecord(c.start_ev, cur_stream()));
    VDF_CUDA_CHECK(cudaStreamWaitEvent(s.stream, c.start_ev, 0));
    if (n) VDF_CUDA_CHECK(cudaMemcpyAsync(s.d_scalars, scalars32_host, n * 32, cudaMemcpyHostToDevice, s.stream));
    msm_on_device(g, 0, s.d_scalars, n, s.d_out, true, s.stream);
    VDF_CUDA_CHECK(cudaMemcpyAsync(out_point96_host, s.d_out, sizeof(jac_t), cudaMemcpyDeviceToHost, s.stream));
    VDF_CUDA_CHECK(cudaEventRecord(s.done, s.stream));
    s.busy = true;
  });
}

int vdfgpu_msm_wait(int slot) {
  return guarded([&] {
    if (slot < 0 || slot >= VDF_ASYNC_SLOTS) throw ArgError("msm_wait: slot out of range");
    require_ready();
    AsyncSlot& s = ctx().slots[slot];
    if (!s.busy) throw StateError("msm_wait: nothing in flight in this slot");
    t_wait_ev = s.done;   // waited for after the context mutex is released
    s.busy = false;
  });
}

int vdfgpu_msm_dev(vdfgpu_gens* g, const void* scalars32_dev, size_t n, void* out_point96_dev) {
  return guarded([&] {
    if (!g || !out_point96_dev || (n && !scalars32_dev)) throw ArgError("msm_dev: null pointer");
    require_ready();
    msm_on_device(g, 0, reinterpret_cast<const fe*>(scalars32_dev), n, reinterpret_cast<jac_t*>(out_point96_dev),
                  true);
  });
}

int vdfgpu_msm_batch_dev(vdfgpu_gens* g, const void* const* scalars32_dev, const size_t* lens, uint32_t k,
                         void* out_points96_dev) {
  return guarded([&] {
    if (!g || !scalars32_dev || !lens || !out_points96_dev) throw ArgError("msm_batch_dev: null pointer");
    require_ready();
    msm_batch_on_device(g, reinterpret_cast<const fe* const*>(scalars32_dev), lens, k,
                        reinterpret_cast<jac_t*>(out_points96_dev));
  });
}

int vdfgpu_msm_range_dev(vdfgpu_gens* g, size_t first, const void* scalars32_dev, size_t n,
                         void* out_point96_dev) {
  return guarded([&] {
    if (!g || !out_point96_dev || (n && !scalars32_dev)) throw ArgError("msm_range_dev: null pointer");
    if (g->flags & VDFGPU_GENS_TABLE && first != 0)
      throw ArgError("msm_range_dev: table-mode sets are sharded by creating one set per rank");
    require_ready();
    msm_on_device(g, first, reinterpret_cast<const fe*>(scalars32_dev), n,
                  reinterpret_cast<jac_t*>(out_point96_dev), true);
  });
}

int vdfgpu_point_sum(int curve, const void* points96_host, size_t k, void* out_point96_host) {
  return guarded([&] {
    if (!out_point96_host || (k && !points96_host)) throw ArgError("point_sum: null pointer");
    with_curve(curve, "point_sum", [&](auto C, auto, auto) {
      require_ready();
      CudaLaunch L = api_launch(cur_stream());
      DevBuf<jac_t> in(k ? k : 1, cur_stream());
      DevBuf<jac_t> res(1, cur_stream());
      h2d(in.p, points96_host, k * sizeof(jac_t), cur_stream());
      L.run<32>(32, JacSumFn<decltype(C)>{in.p, (uint32_t)k, res.p});
      d2h(out_point96_host, res.p, sizeof(jac_t), cur_stream());
      sync_after_unlock(cur_stream());
    });
  });
}

int vdfgpu_point_normalise_host(int curve, void* points96_host, size_t count) {
  try {   // host arithmetic only: no device, no lock
    hostfield::coord_mod(curve);   // ArgError for an unknown curve
    if (count && !points96_host) throw ArgError("point_normalise_host: null pointer");
  } catch (const ArgError& e) {
    set_error(e.what());
    return VDFGPU_ERR_ARG;
  }
  for (size_t k = 0; k < count;) {   // 16 points per inversion
    uint8_t* pts[16];
    size_t m = 0;
    for (; m < 16 && k < count; m++, k++) pts[m] = reinterpret_cast<uint8_t*>(points96_host) + 96 * k;
    if (m == 1) hostfield::normalise(pts[0], curve);
    else hostfield::normalise_batch(pts, m, curve);
  }
  return VDFGPU_OK;
}

int vdfgpu_point_sum_dev(int curve, const void* points96_dev, size_t k, void* out_point96_dev) {
  return guarded([&] {
    if (!out_point96_dev || (k && !points96_dev)) throw ArgError("point_sum_dev: null pointer");
    with_curve(curve, "point_sum_dev", [&](auto C, auto, auto) {
      require_ready();
      CudaLaunch L = api_launch(cur_stream());
      L.run<32>(32, JacSumFn<decltype(C)>{reinterpret_cast<const jac_t*>(points96_dev), (uint32_t)k,
                                          reinterpret_cast<jac_t*>(out_point96_dev)});
    });
  });
}

// ---- drop-in cache behind mult_pippenger_{pallas,vesta} ----------------------------------------------------
// pasta-msm's entry point receives the points with every call, but its only caller on this path, nova's
// commit(), passes the SAME generators every time (fixed for the life of PublicParams, src/nova/proof.rs:232-237;
// commit(W) and commit(T) use prefixes of one Vec).  So the first call with a new (curve, host pointer) uploads and
// repacks the points, builds the window table and keeps the set resident; later calls with that pointer and
// npoints <= the cached length upload only the scalars and take the same path as vdfgpu_msm().
// A cached set is trusted only while a sample of the caller's points still matches byte for byte (x, y and the
// infinity flag of ~530 points: the first and last 8 and an even stride); VDFGPU_DROPIN_VERIFY=full hashes every
// point on every call instead (exact, ~70 ms per 2^22 points of host time), =off trusts pointer + length.
// VDFGPU_DROPIN_CACHE=0 disables the cache (every call is one-shot), VDFGPU_DROPIN_ENTRIES bounds it (LRU, default 4).
static constexpr size_t DROPIN_MIN_POINTS = 1024;   // below this the one-shot path is as fast

static std::vector<size_t> dropin_sample_indices(size_t n) {
  std::vector<size_t> idx;
  const size_t edge = 8, strided = 512;
  for (size_t i = 0; i < edge && i < n; i++) idx.push_back(i);
  const size_t step = n / strided ? n / strided : 1;
  for (size_t i = edge; i + edge < n; i += step) idx.push_back(i);
  for (size_t i = n > 2 * edge ? n - edge : (n > edge ? edge : n); i < n; i++) idx.push_back(i);
  return idx;
}

static uint64_t dropin_full_hash(const uint8_t* pts72, size_t n) {
  uint64_t h = 0x9e3779b97f4a7c15ull;
  for (size_t i = 0; i < n; i++) {
    uint64_t w[9];
    std::memcpy(w, pts72 + i * 72, 72);
    w[8] &= 0xffull;   // the 7 padding bytes of the repr(C) struct are indeterminate
    for (int k = 0; k < 9; k++) {
      h ^= w[k];
      h *= 0xff51afd7ed558ccdull;
      h ^= h >> 29;
    }
  }
  return h;
}

static int dropin_verify_mode() {   // 0 off, 1 sample, 2 full
  const char* s = std::getenv("VDFGPU_DROPIN_VERIFY");
  if (!s) return 1;
  if (!std::strcmp(s, "off")) return 0;
  if (!std::strcmp(s, "full")) return 2;
  return 1;
}

static void dropin_drop(DropinEntry& e) {
  if (e.gens) GensRelease()(e.gens);
  e.gens = nullptr;
}

static void dropin_clear_locked() {
  Context& c = ctx();
  if (c.dropin.empty()) return;
  if (c.ready) cudaDeviceSynchronize();
  for (auto& e : c.dropin) dropin_drop(e);
  c.dropin.clear();
}

static bool dropin_matches(const DropinEntry& e, int curve, const uint8_t* pts72, size_t npoints, int mode) {
  if (e.curve != curve || e.host_ptr != pts72 || npoints > e.n) return false;
  if (mode == 0) return true;
  if (mode == 2) return npoints == e.n && dropin_full_hash(pts72, npoints) == e.full_hash;
  for (size_t k = 0; k < e.sample_idx.size(); k++) {
    const size_t i = e.sample_idx[k];
    if (i >= npoints) break;
    if (std::memcmp(pts72 + i * 72, &e.sample_bytes[k * 65], 65) != 0) return false;
  }
  return true;
}

// resident generator set for this call's points, or nullptr: take the one-shot path
static vdfgpu_gens* dropin_lookup(int curve, const void* points, size_t npoints) {
  Context& c = ctx();
  if (npoints < DROPIN_MIN_POINTS || env_long("VDFGPU_DROPIN_CACHE", 1, 0, 1) == 0) return nullptr;
  const uint8_t* pts72 = reinterpret_cast<const uint8_t*>(points);
  const int mode = dropin_verify_mode();
  for (size_t k = 0; k < c.dropin.size(); k++) {
    DropinEntry& e = c.dropin[k];
    if (e.curve != curve || e.host_ptr != points) continue;
    if (dropin_matches(e, curve, pts72, npoints, mode)) {
      e.last_use = ++c.tick;
      c.dropin_hits++;
      return e.gens;
    }
    // same address, other contents or a longer slice: the cached set is stale
    cudaDeviceSynchronize();
    dropin_drop(e);
    c.dropin.erase(c.dropin.begin() + k);
    break;
  }
  c.dropin_misses++;
  const size_t max_entries = (size_t)env_long("VDFGPU_DROPIN_ENTRIES", 4, 1, 64);
  while (c.dropin.size() >= max_entries) {
    size_t lru = 0;
    for (size_t i = 1; i < c.dropin.size(); i++)
      if (c.dropin[i].last_use < c.dropin[lru].last_use) lru = i;
    cudaDeviceSynchronize();
    dropin_drop(c.dropin[lru]);
    c.dropin.erase(c.dropin.begin() + lru);
  }
  // window table when it fits comfortably (W levels of 64 B per point), plain resident points otherwise
  uint32_t flags = VDFGPU_GENS_TABLE;
  size_t free_b = 0, total_b = 0;
  VDF_CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
  const uint32_t c_bits = msm_pick_c(npoints, true);
  if ((uint64_t)msm_windows(c_bits) * npoints >= (1ull << 31) ||
      (size_t)msm_windows(c_bits) * npoints * sizeof(affine_t) > free_b / 3)
    flags = 0;
  GensPtr g = gens_upload(curve, points, npoints, flags, 0, cur_stream());
  DropinEntry e;
  e.curve = curve;
  e.host_ptr = points;
  e.n = npoints;
  e.sample_idx = dropin_sample_indices(npoints);
  e.sample_bytes.resize(e.sample_idx.size() * 65);
  for (size_t k = 0; k < e.sample_idx.size(); k++)
    std::memcpy(&e.sample_bytes[k * 65], pts72 + e.sample_idx[k] * 72, 65);
  if (mode == 2) e.full_hash = dropin_full_hash(pts72, npoints);
  e.gens = g.release();
  e.last_use = ++c.tick;
  c.dropin.push_back(std::move(e));
  return c.dropin.back().gens;
}

static void mult_pippenger_body(int curve, void* out, const void* points, size_t npoints, const void* scalars,
                                bool is_mont) {
  require_ready();
  cudaStream_t st = cur_stream();
  if (workspaces_enabled()) {
    if (vdfgpu_gens* cached = dropin_lookup(curve, points, npoints)) {
      Workspace* ws = staging_for(st, npoints);
      h2d_scalars(ws->stage_sc, scalars, npoints * 32, st);
      const bool hn = host_normalise_wanted(cached);
      msm_on_device(cached, 0, ws->stage_sc, npoints, ws->stage_out, is_mont, nullptr, hn);
      d2h(out, ws->stage_out, sizeof(jac_t), st);
      sync_after_unlock(st);
      if (hn) normalise_after_sync(out, 1, curve);
      return;
    }
  }
  DevBuf<fe> sc(npoints, st);
  DevBuf<jac_t> res(1, st);
  h2d(sc.p, scalars, npoints * 32, st);
  if (vdfgpu_gens* cached = workspaces_enabled() ? nullptr : dropin_lookup(curve, points, npoints)) {
    msm_on_device(cached, 0, sc.p, npoints, res.p, is_mont);
  } else {
    vdfgpu_gens g;
    g.curve = curve;
    g.n = npoints;
    g.flags = 0;
    g.W = 1;
    CudaLaunch L = api_launch(st);
    DevBuf<uint8_t> raw(npoints * 72, st);
    DevBuf<affine_t> pts(npoints, st);
    h2d(raw.p, points, npoints * 72, st);
    L.run<256>(npoints, RepackFn{raw.p, pts.p});
    g.pts = pts.p;
    msm_on_device(&g, 0, sc.p, npoints, res.p, is_mont);
  }
  d2h(out, res.p, sizeof(jac_t), st);
  sync_after_unlock(st);
}

static void mult_pippenger(int curve, void* out, const void* points, size_t npoints, const void* scalars,
                           bool is_mont) {
  // pasta-msm's entry point is infallible (void) and its Rust wrapper asserts points.len() == scalars.len().
  // Argument misuse: say so and return the identity.  A CUDA failure (typically out of memory): drop every cached
  // set and workspace, trim the pool and retry once; only a second failure aborts, as the reference would panic.
  if (!out) {
    std::fprintf(stderr, "mult_pippenger: null output pointer\n");
    return;
  }
  if (npoints == 0 || !points || !scalars) {
    if (npoints) std::fprintf(stderr, "mult_pippenger: null points/scalars with npoints = %zu; returning the identity\n", npoints);
    std::memset(out, 0, 96);
    return;
  }
  int rc = guarded([&] { mult_pippenger_body(curve, out, points, npoints, scalars, is_mont); });
  if (rc == VDFGPU_ERR_CUDA) {
    std::fprintf(stderr, "mult_pippenger: %s -- releasing cached sets and workspaces, retrying once\n", vdfgpu_last_error());
    guarded([&] {
      cudaGetLastError();
      dropin_clear_locked();
      trim_locked();
    });
    rc = guarded([&] { mult_pippenger_body(curve, out, points, npoints, scalars, is_mont); });
  }
  if (rc != VDFGPU_OK) {
    std::fprintf(stderr, "mult_pippenger: %s\n", vdfgpu_last_error());
    std::abort();
  }
}

void mult_pippenger_pallas(void* out, const void* points, size_t npoints, const void* scalars, bool is_mont) {
  mult_pippenger(VDFGPU_PALLAS, out, points, npoints, scalars, is_mont);
}

void mult_pippenger_vesta(void* out, const void* points, size_t npoints, const void* scalars, bool is_mont) {
  mult_pippenger(VDFGPU_VESTA, out, points, npoints, scalars, is_mont);
}

int vdfgpu_dropin_cache_clear(void) {
  return guarded([&] { dropin_clear_locked(); });
}

int vdfgpu_dropin_cache_stats(uint64_t* hits, uint64_t* misses, uint64_t* entries) {
  return guarded([&] {
    Context& c = ctx();
    if (hits) *hits = c.dropin_hits;
    if (misses) *misses = c.dropin_misses;
    if (entries) *entries = c.dropin.size();
  });
}

// ---- batched MinRoot verification -----------------------------------------------------------------------
int vdfgpu_minroot_check_batch_dev(int field, const void* results_dev, const void* originals_dev,
                                   const uint64_t* t_each_dev, uint64_t t_uniform, size_t n,
                                   uint8_t* ok_out_dev) {
  return guarded([&] {
    with_field(field, "minroot_check", [&](auto f) {
      if (n && (!results_dev || !originals_dev || !ok_out_dev)) throw ArgError("minroot_check: null pointer");
      require_ready();
      CudaLaunch L = api_launch(cur_stream());
      minroot_check_dispatch<decltype(f)>(L, results_dev, originals_dev, t_each_dev, t_uniform, n, ok_out_dev);
    });
  });
}

int vdfgpu_minroot_check_batch(int field, const void* results_host, const void* originals_host,
                               const uint64_t* t_each, uint64_t t_uniform, size_t n, uint8_t* ok_out_host) {
  return guarded([&] {
    with_field(field, "minroot_check", [&](auto f) {
      if (n && (!results_host || !originals_host || !ok_out_host)) throw ArgError("minroot_check: null pointer");
      if (n == 0) return;
      require_ready();
      CudaLaunch L = api_launch(cur_stream());
      DevBuf<state_t> res(n, cur_stream()), orig(n, cur_stream());
      DevBuf<uint64_t> tt(t_each ? n : 1, cur_stream());
      DevBuf<uint8_t> ok(n, cur_stream());
      h2d(res.p, results_host, n * sizeof(state_t), cur_stream());
      h2d(orig.p, originals_host, n * sizeof(state_t), cur_stream());
      if (t_each) h2d(tt.p, t_each, n * 8, cur_stream());
      minroot_check_dispatch<decltype(f)>(L, res.p, orig.p, t_each ? tt.p : nullptr, t_uniform, n, ok.p);
      d2h(ok_out_host, ok.p, n, cur_stream());
      sync_after_unlock(cur_stream());
    });
  });
}

int vdfgpu_minroot_inverse_eval_batch(int field, const void* results_host, uint64_t t, size_t n,
                                      void* out_host) {
  return guarded([&] {
    with_field(field, "minroot_inverse_eval", [&](auto f) {
      if (n && (!results_host || !out_host)) throw ArgError("minroot_inverse_eval: null pointer");
      if (n == 0) return;
      require_ready();
      CudaLaunch L = api_launch(cur_stream());
      DevBuf<state_t> res(n, cur_stream()), out(n, cur_stream());
      h2d(res.p, results_host, n * sizeof(state_t), cur_stream());
      L.run<128>(n, MinRootInverseEvalFn<decltype(f)>{res.p, t, out.p});
      d2h(out_host, out.p, n * sizeof(state_t), cur_stream());
      sync_after_unlock(cur_stream());
    });
  });
}

int vdfgpu_minroot_witness_batch(int field, const void* results_host, uint64_t t, size_t n, void* out_host) {
  return guarded([&] {
    with_field(field, "minroot_witness", [&](auto f) {
      if (n && (!results_host || !out_host)) throw ArgError("minroot_witness: null pointer");
      if (n == 0) return;
      require_ready();
      CudaLaunch L = api_launch(cur_stream());
      const size_t per = 4 * (size_t)t + 1;
      DevBuf<state_t> res(n, cur_stream());
      DevBuf<fe> out(n * per, cur_stream());
      h2d(res.p, results_host, n * sizeof(state_t), cur_stream());
      L.run<128>(n, MinRootWitnessFn<decltype(f)>{res.p, t, out.p});
      d2h(out_host, out.p, n * per * 32, cur_stream());
      sync_after_unlock(cur_stream());
    });
  });
}

// ---- probes ---------------------------------------------------------------------------------------------
int vdfgpu_field_mul_batch(int field, const void* a_host, const void* b_host, size_t n, uint32_t iters,
                           void* out_host) {
  return guarded([&] {
    with_field(field, "field_mul_batch", [&](auto f) {
      if (n && (!a_host || !b_host || !out_host)) throw ArgError("field_mul_batch: null pointer");
      if (n == 0) return;
      require_ready();
      CudaLaunch L = api_launch(cur_stream());
      DevBuf<fe> a(n, cur_stream()), b(n, cur_stream()), o(n, cur_stream());
      h2d(a.p, a_host, n * 32, cur_stream());
      h2d(b.p, b_host, n * 32, cur_stream());
      L.run<256>(n, FieldMulFn<decltype(f)>{a.p, b.p, o.p, iters});
      d2h(out_host, o.p, n * 32, cur_stream());
      sync_after_unlock(cur_stream());
    });
  });
}

int vdfgpu_imad_peak(double* mul32_per_s_wide, double* imad_per_s_lo, double* iadd3_per_s) {
  return guarded([&] {
    require_ready();
    DevBuf<uint32_t> sink(4, cur_stream());
    double w = probe_rate<0>(cur_stream(), sink.p);
    double l = probe_rate<1>(cur_stream(), sink.p);
    double a = probe_rate<2>(cur_stream(), sink.p);
    ctx().launches += 9;
    if (mul32_per_s_wide) *mul32_per_s_wide = w;
    if (imad_per_s_lo) *imad_per_s_lo = l;
    if (iadd3_per_s) *iadd3_per_s = a;
  });
}

#pragma GCC visibility pop
}  // extern "C"
