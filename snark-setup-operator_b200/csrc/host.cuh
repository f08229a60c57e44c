// Host-side plumbing shared by the per-curve translation units and the C ABI (abi.cu):
// error strings, Phase1Parameters layout arithmetic, per-call CUDA context (own streams and
// stream-ordered scratch, so every ABI call is re-entrant — SURVEY.md §8b "Threading").
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <chrono>
#include <cstdlib>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/sso_b200.h"

namespace sso {


inline void set_err(char* err, size_t cap, const char* fmt, ...) {
  if (!err || cap == 0) return;
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(err, cap, fmt, ap);
  va_end(ap);
}

#define CUDA_TRY(expr)                                                                              \
  do {                                                                                              \
    cudaError_t e_ = (expr);                                                                        \
    if (e_ != cudaSuccess) {                                                                        \
      set_err(err, errcap, "CUDA error %s at %s:%d (%s)", cudaGetErrorName(e_), __FILE__, __LINE__, \
              cudaGetErrorString(e_));                                                              \
      return SSO_E_CUDA;                                                                            \
    }                                                                                               \
  } while (0)

struct CurveSizes { uint64_t g1c, g1u, g2c, g2u, fr; };
inline bool curve_sizes(uint32_t curve, CurveSizes& s) {
  switch (curve) {
    case SSO_CURVE_BLS12_377: s = {48, 96, 96, 192, 32}; return true;
    case SSO_CURVE_BW6_761: s = {96, 192, 96, 192, 48}; return true;
    case SSO_CURVE_MNT4_753: s = {95, 190, 190, 380, 95}; return true;
    case SSO_CURVE_MNT6_753: s = {95, 190, 285, 570, 95}; return true;
  }
  return false;
}

// Phase1Parameters arithmetic (SURVEY.md Appendix A.4)
struct P1Layout {
  uint64_t powers_length, powers_g1_length, g1n, on, acc_size, contrib_size, pk_size, num_chunks, start;
  uint64_t off_u[6], off_c[6];   // tauG1, tauG2, alphaG1, betaG1, betaG2, end
  CurveSizes cs;
};
inline int p1_layout(const sso_p1_params_t* p, P1Layout& L, char* err, size_t errcap) {
  if (!p) { set_err(err, errcap, "null parameters"); return SSO_E_ARG; }
  if (!curve_sizes(p->curve, L.cs)) { set_err(err, errcap, "unknown curve %u", p->curve); return SSO_E_ARG; }
  if (p->proving_system != SSO_PROVING_GROTH16) { set_err(err, errcap, "only the Groth16 proving system is supported"); return SSO_E_ARG; }
  if (p->power == 0 || p->power > 32) { set_err(err, errcap, "power out of range"); return SSO_E_ARG; }
  L.powers_length = 1ull << p->power;
  L.powers_g1_length = (1ull << (p->power + 1)) - 1;
  if (p->contribution_mode == SSO_MODE_FULL) {
    L.start = 0; L.g1n = L.powers_g1_length; L.on = L.powers_length; L.num_chunks = 1;
  } else {
    if (p->chunk_size == 0) { set_err(err, errcap, "chunk_size must be positive in chunked mode"); return SSO_E_ARG; }
    L.start = p->chunk_index * p->chunk_size;
    L.g1n = L.start >= L.powers_g1_length ? 0 : (L.powers_g1_length - L.start < p->chunk_size ? L.powers_g1_length - L.start : p->chunk_size);
    L.on = L.start >= L.powers_length ? 0 : (L.powers_length - L.start < p->chunk_size ? L.powers_length - L.start : p->chunk_size);
    L.num_chunks = (L.powers_g1_length + p->chunk_size - 1) / p->chunk_size;
  }
  L.pk_size = 3 * L.cs.g2u + 6 * L.cs.g1u;
  auto fill = [&](uint64_t* off, uint64_t g1, uint64_t g2) {
    off[0] = 64; off[1] = off[0] + L.g1n * g1; off[2] = off[1] + L.on * g2; off[3] = off[2] + L.on * g1;
    off[4] = off[3] + L.on * g1; off[5] = off[4] + g2;
  };
  fill(L.off_u, L.cs.g1u, L.cs.g2u);
  fill(L.off_c, L.cs.g1c, L.cs.g2c);
  L.acc_size = L.off_u[5];
  L.contrib_size = L.off_c[5] + L.pk_size;
  return SSO_OK;
}

inline const char* status_text(uint32_t code) {
  switch (code) {
    case 1: return "field element is not canonical (>= modulus)";
    case 2: return "invalid point flags";
    case 3: return "point is not on the curve";
    case 4: return "point at infinity";
    case 5: return "point is not in the prime-order subgroup";
  }
  return "unknown";
}

// Per-kernel launch accounting (always on) and optional CUDA-event timing on the launching stream
// (sso_profile_enable) — the source of bench.py's roofline.achieved and gpu_launches.
enum ProfKind { PK_TAU_TABLES = 0, PK_BATCH_EXP_G1, PK_BATCH_EXP_G2, PK_NORMALIZE_G1, PK_NORMALIZE_G2, PK_REENCODE_G1,
                PK_REENCODE_G2, PK_FILL, PK_MSM, PK_OTHER, PK_BATCH_EXP_CHUNK, PK_NORMALIZE_CHUNK, PK_COUNT };
struct ProfSlot { std::atomic<uint64_t> launches{0}; std::atomic<uint64_t> ns{0}; std::atomic<uint64_t> elems{0}; };
extern ProfSlot g_prof[PK_COUNT];
extern std::atomic<int> g_prof_enabled;

// RAII: device selection + streams + stream-ordered scratch; one per ABI call (re-entrant)
struct Ctx {
  int dev = -1, prev = -1;
  bool aliased = false;
  cudaStream_t s[3] = {nullptr, nullptr, nullptr};    // s[2] (when asked for) has the highest priority: short latency-critical kernels
  bool owned[3] = {false, false, false};
  std::vector<void*> allocs;
  std::vector<std::vector<uint32_t>> staging;     // host copies that must outlive async H2D
  struct Timed { int kind; cudaEvent_t e0, e1; };
  std::vector<Timed> timed;
  char* err; size_t errcap;
  // SSO_TRACE=1: host-side timeline of the call on stderr (debugging aid)
  bool trace = false;
  std::chrono::steady_clock::time_point t_start, t_last;
  void mark(const char* what) {
    if (!trace) return;
    auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[sso trace] %-28s +%8.3f ms (total %8.3f ms)\n", what,
            std::chrono::duration<double, std::milli>(now - t_last).count(),
            std::chrono::duration<double, std::milli>(now - t_start).count());
    t_last = now;
  }
  Ctx(char* e, size_t c) : err(e), errcap(c) {
    const char* tr = getenv("SSO_TRACE");
    trace = tr && tr[0] == '1';
    t_start = t_last = std::chrono::steady_clock::now();
  }
  int init(int device, int nstreams = 1) {
    int cnt = 0;
    if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt == 0) {
      set_err(err, errcap, "no CUDA device available (this library has no CPU fallback)");
      return SSO_E_CUDA;
    }
    if (device < 0 || device >= cnt) { set_err(err, errcap, "device %d out of range (have %d)", device, cnt); return SSO_E_ARG; }
    cudaGetDevice(&prev);
    CUDA_TRY(cudaSetDevice(device));
    dev = device;
    // keep stream-ordered scratch cached in the device's default pool between calls: with the default
    // release threshold (0) every synchronisation hands the memory back to the driver and the next
    // call pays tens of milliseconds to map it again (measured: 5-80 ms per call on B200)
    static std::atomic<uint64_t> pool_configured{0};
    if (device < 64 && !(pool_configured.load() & (1ull << device))) {
      cudaMemPool_t pool;
      if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        uint64_t keep = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
      }
      pool_configured.fetch_or(1ull << device);
    }
    // profiling mode 2 serialises the call on ONE stream so that per-kernel event times are not inflated by
    // kernels of the other stream sharing the SMs (used for the roofline pass of bench.py)
    aliased = nstreams > 1 && g_prof_enabled.load(std::memory_order_relaxed) == 2;
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);                 // hi = numerically lowest = highest priority
    for (int i = 0; i < (aliased ? 1 : nstreams) && i < 3; i++) {
      if (i == 2) CUDA_TRY(cudaStreamCreateWithPriority(&s[i], cudaStreamNonBlocking, hi));
      else CUDA_TRY(cudaStreamCreateWithFlags(&s[i], cudaStreamNonBlocking));
      owned[i] = true;
    }
    if (aliased) for (int i = 1; i < nstreams && i < 3; i++) s[i] = s[0];
    mark("init: device + streams");
    return SSO_OK;
  }
  int alloc(void** p, size_t bytes, int si = 0) {
    CUDA_TRY(cudaMallocAsync(p, bytes ? bytes : 16, s[si]));
    allocs.push_back(*p);
    return SSO_OK;
  }
  // between the pieces of a streamed call: hand the scratch of the finished piece back to the pool (stream-ordered)
  // and drop the host staging copies; the streams stay
  int recycle() {
    for (auto& st : s) if (st) CUDA_TRY(cudaStreamSynchronize(st));
    resolve_timings();
    for (void* p : allocs) cudaFreeAsync(p, s[0]);
    allocs.clear();
    staging.clear();
    return SSO_OK;
  }
  // stream-ordered release of the scratch allocated since allocs.size() was `from`: a long piece hands back what one of its
  // steps needed before the next step allocates (the pool reuses it)
  void release(size_t from) {
    for (size_t i = from; i < allocs.size(); i++) cudaFreeAsync(allocs[i], s[0]);
    allocs.resize(from);
  }
  // make stream `to` wait for everything enqueued so far on stream `from`
  int fork(int from, int to) {
    cudaEvent_t ev;
    CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    CUDA_TRY(cudaEventRecord(ev, s[from]));
    CUDA_TRY(cudaStreamWaitEvent(s[to], ev, 0));
    CUDA_TRY(cudaEventDestroy(ev));
    return SSO_OK;
  }
  // bracket a kernel launch: counts it, and times it with events on its own stream when profiling is on
  void begin(int kind, int si, uint64_t elems) {
    g_prof[kind].launches.fetch_add(1, std::memory_order_relaxed);
    g_prof[kind].elems.fetch_add(elems, std::memory_order_relaxed);
    if (g_prof_enabled.load(std::memory_order_relaxed)) {
      Timed t{kind, nullptr, nullptr};
      cudaEventCreate(&t.e0);
      cudaEventCreate(&t.e1);
      cudaEventRecord(t.e0, s[si]);
      timed.push_back(t);
    }
  }
  void end(int si) {
    if (!timed.empty() && g_prof_enabled.load(std::memory_order_relaxed)) cudaEventRecord(timed.back().e1, s[si]);
  }
  void resolve_timings() {
    for (auto& t : timed) {
      float ms = 0;
      if (cudaEventSynchronize(t.e1) == cudaSuccess && cudaEventElapsedTime(&ms, t.e0, t.e1) == cudaSuccess)
        g_prof[t.kind].ns.fetch_add((uint64_t)(ms * 1e6), std::memory_order_relaxed);
      cudaEventDestroy(t.e0);
      cudaEventDestroy(t.e1);
    }
    timed.clear();
  }
  ~Ctx() {
    if (dev >= 0) {
      for (auto& st : s) if (st) cudaStreamSynchronize(st);
      resolve_timings();
      mark("dtor: streams drained");
      for (void* p : allocs) cudaFreeAsync(p, s[0]);
      for (int i = 0; i < 3; i++) if (s[i] && owned[i]) { cudaStreamSynchronize(s[i]); cudaStreamDestroy(s[i]); }
      if (prev >= 0) cudaSetDevice(prev);
      mark("dtor: freed + destroyed");
    }
  }
};

inline uint32_t div_up(uint64_t a, uint64_t b) { return (uint32_t)((a + b - 1) / b); }

// canonical little-endian scalar bytes -> zero-padded words on the device
inline int upload_scalar(Ctx& c, const uint8_t* bytes, size_t nbytes, size_t nwords, uint32_t** d_out, int si, char* err, size_t errcap) {
  c.staging.emplace_back(nwords, 0u);
  std::vector<uint32_t>& w = c.staging.back();    // kept alive by the context until the call ends
  if (bytes) memcpy(w.data(), bytes, nbytes);
  else w[0] = 1;
  int rc = c.alloc((void**)d_out, nwords * 4, si);
  if (rc) return rc;
  CUDA_TRY(cudaMemcpyAsync(*d_out, w.data(), nwords * 4, cudaMemcpyHostToDevice, c.s[si]));
  return SSO_OK;
}

// status words written by kernels: [0] code, [1] element index inside its vector, [2] vector index
static constexpr size_t STATUS_BYTES = 16;
// a zeroed status buffer on stream si; `sync` drains that stream before the call goes on
inline int status_buffer(Ctx& c, uint32_t** d_status, int si, bool sync, char* err, size_t errcap) {
  int rc = c.alloc((void**)d_status, STATUS_BYTES, si);
  if (rc) return rc;
  CUDA_TRY(cudaMemsetAsync(*d_status, 0, STATUS_BYTES, c.s[si]));
  if (sync) CUDA_TRY(cudaStreamSynchronize(c.s[si]));
  return SSO_OK;
}
inline int check_status(Ctx& c, uint32_t* d_status, const char* what, char* err, size_t errcap) {
  uint32_t h[4] = {0, 0, 0, 0};
  CUDA_TRY(cudaMemcpy(h, d_status, STATUS_BYTES, cudaMemcpyDeviceToHost));
  if (h[0] != 0) {
    set_err(err, errcap, "%s: %s (vector %u, element %u)", what, status_text(h[0]), h[2], h[1]);
    return h[0] == 5u ? SSO_E_VERIFY : SSO_E_INPUT;
  }
  return SSO_OK;
}

inline int sync_all(Ctx& c, char* err, size_t errcap) {
  c.mark("launches enqueued");
  for (auto st : c.s) if (st) CUDA_TRY(cudaStreamSynchronize(st));
  c.mark("streams synchronized");
  c.resolve_timings();
  return SSO_OK;
}


}  // namespace sso
