// Streaming of vectors that do not fit one launch (or one GPU): the Full-mode accumulator the beacon contribution and
// the final ratio verification work on (reference src/bin/verify_transcript.rs:603-607, 675-696, 746-776, 811-822;
// src/bin/control.rs:564-591, 792-873) has 2^(p+1) - 1 + 3 * 2^p points — 64 GB at BW6-761 2^26.  Every vector is cut into
// pieces of at most `batch_size` elements (Phase1Parameters::batch_size, reference src/bin/new_setup.rs:259); host
// workers pull pieces from a queue, each on its own stream (copies of one piece overlap the kernels of another), and
// the workers are spread over the devices of the call.  Pieces are independent for the contribution (the tau table of
// a piece starts at tau^(start + offset)); the random-linear-combination MSMs of the verification leave one partial
// pair per piece, the partial pairs of a device are summed on that device, and the per-device sums are exchanged with
// ONE all-gather (NCCL over NVLink) followed by a point addition — the only collective of the path (SURVEY.md §8e).
//
// Participants of the exchange are either the devices of this process (sso_*_file(devices, ndev): ncclCommInitAll)
// or the ranks of a process group with one GPU each (sso_dist_init: ncclCommInitRank with an id the caller broadcast,
// e.g. over torch.distributed).  NCCL is loaded at run time (dlopen of the libnccl.so.2 the process already holds,
// else the system one), so the library loads on hosts without it and single-GPU calls never touch it.
#pragma once
#include <dlfcn.h>
#include <nccl.h>
#include <functional>
#include <map>

namespace sso {

// ---------------------------------------------------------------------------------------------
// NCCL through dlopen
// ---------------------------------------------------------------------------------------------
struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  ncclResult_t (*GetVersion)(int*) = nullptr;
};
inline const NcclApi* nccl_api(char* err, size_t errcap) {
  static NcclApi api;
  static std::once_flag once;
  static std::string why;
  std::call_once(once, [] {
    const char* names[] = {"libnccl.so.2", "libnccl.so", "/usr/lib/x86_64-linux-gnu/libnccl.so.2"};
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);      // the copy torch (or the host program) holds
    for (int i = 0; !h && i < 3; i++) h = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
    if (!h) { why = "NCCL is not available (dlopen libnccl.so.2 failed)"; return; }
    api.handle = h;
#define SSO_NCCL_SYM(field, name) *(void**)(&api.field) = dlsym(h, name); if (!api.field) { why = std::string("NCCL symbol missing: ") + name; api.handle = nullptr; return; }
    SSO_NCCL_SYM(GetUniqueId, "ncclGetUniqueId")
    SSO_NCCL_SYM(CommInitRank, "ncclCommInitRank")
    SSO_NCCL_SYM(CommInitAll, "ncclCommInitAll")
    SSO_NCCL_SYM(CommDestroy, "ncclCommDestroy")
    SSO_NCCL_SYM(AllGather, "ncclAllGather")
    SSO_NCCL_SYM(AllReduce, "ncclAllReduce")
    SSO_NCCL_SYM(GroupStart, "ncclGroupStart")
    SSO_NCCL_SYM(GroupEnd, "ncclGroupEnd")
    SSO_NCCL_SYM(GetErrorString, "ncclGetErrorString")
    SSO_NCCL_SYM(GetVersion, "ncclGetVersion")
#undef SSO_NCCL_SYM
  });
  if (!api.handle) { set_err(err, errcap, "%s", why.c_str()); return nullptr; }
  return &api;
}
#define NCCL_TRY(api, expr)                                                                          \
  do {                                                                                               \
    ncclResult_t r_ = (expr);                                                                        \
    if (r_ != ncclSuccess) {                                                                         \
      set_err(err, errcap, "NCCL error at %s:%d: %s", __FILE__, __LINE__, (api)->GetErrorString(r_)); \
      return SSO_E_CUDA;                                                                             \
    }                                                                                                \
  } while (0)

// one GPU per process, several processes (torchrun): the communicator of the process group
struct DistState {
  bool on = false;
  int rank = 0, world = 1, device = 0;
  ncclComm_t comm = nullptr;
  uint64_t collectives = 0;       // all-gathers issued so far (reported by sso_dist_stats)
};
inline DistState& dist_state() { static DistState d; return d; }
inline std::mutex& dist_mutex() { static std::mutex m; return m; }

// communicators over the devices of ONE process, cached per device list (ncclCommInitAll takes ~0.3 s per device)
struct LocalComms { std::vector<int> devices; std::vector<ncclComm_t> comms; };
inline int local_comms(const std::vector<int>& devices, LocalComms** out, char* err, size_t errcap) {
  static std::map<std::vector<int>, LocalComms> cache;
  std::lock_guard<std::mutex> g(dist_mutex());
  auto it = cache.find(devices);
  if (it == cache.end()) {
    const NcclApi* api = nccl_api(err, errcap);
    if (!api) return SSO_E_CUDA;
    LocalComms lc;
    lc.devices = devices;
    lc.comms.resize(devices.size());
    NCCL_TRY(api, api->CommInitAll(lc.comms.data(), (int)devices.size(), devices.data()));
    it = cache.emplace(devices, std::move(lc)).first;
  }
  *out = &it->second;
  return SSO_OK;
}

// ---------------------------------------------------------------------------------------------
// Work queue over pieces: `workers_per_device` host threads per device, each with ONE context (streams live for the
// whole call, scratch is recycled after every piece).  fn(piece index, device slot, ctx, err, errcap).
// ---------------------------------------------------------------------------------------------
struct Participants {
  std::vector<int> devices;       // devices of this process that take part
  // pieces are dealt round-robin over (rank, world) first when the call is a cooperative one of a process group
  int rank = 0, world = 1;
  bool dist = false;
};
// cooperative: the call is made by every rank of the process group on the same files (Full-mode calls, combine,
// transform_ratios); chunk-level calls stay local to the calling rank even when a process group exists
inline int resolve_participants(const int* devices, int ndev, int device, bool cooperative, Participants& P, char* err, size_t errcap) {
  int cnt = 0;
  if (cudaGetDeviceCount(&cnt) != cudaSuccess || cnt <= 0) { set_err(err, errcap, "no CUDA device available (this library has no CPU fallback)"); return SSO_E_CUDA; }
  P.devices.clear();
  DistState& d = dist_state();
  if (cooperative && d.on) {                    // one GPU per rank: the process group decides
    P.devices.push_back(d.device);
    P.rank = d.rank; P.world = d.world; P.dist = true;
    return SSO_OK;
  }
  if (devices && ndev > 0) {
    for (int i = 0; i < ndev; i++) {
      if (devices[i] < 0 || devices[i] >= cnt) { set_err(err, errcap, "device %d out of range (have %d)", devices[i], cnt); return SSO_E_ARG; }
      P.devices.push_back(devices[i]);
    }
  } else if (device < 0) {
    for (int i = 0; i < cnt; i++) P.devices.push_back(i);
  } else {
    if (device >= cnt) { set_err(err, errcap, "device %d out of range (have %d)", device, cnt); return SSO_E_ARG; }
    P.devices.push_back(device);
  }
  return SSO_OK;
}

template <class Fn>
inline int run_pieces(size_t n_pieces, const Participants& P, int workers_per_device, int nstreams, char* err, size_t errcap, Fn fn) {
  if (n_pieces == 0) return SSO_OK;
  std::atomic<size_t> next{0};
  std::atomic<int32_t> first_rc{SSO_OK};
  std::mutex err_lock;
  auto work = [&](int slot) {
    char local[512];
    local[0] = 0;
    Ctx c(local, sizeof local);
    int32_t rc = c.init(P.devices[slot], nstreams);
    while (rc == SSO_OK) {
      size_t i = next.fetch_add(1);
      if (i >= n_pieces || first_rc.load() != SSO_OK) break;
      if ((int)(i % (size_t)P.world) != P.rank) continue;            // another rank's piece
      rc = fn(i, slot, c, local, sizeof local);
      if (rc == SSO_OK) rc = c.recycle();
    }
    if (rc != SSO_OK) {
      std::lock_guard<std::mutex> g(err_lock);
      if (first_rc.load() == SSO_OK) { first_rc.store(rc); set_err(err, errcap, "%s", local); }
    }
  };
  std::vector<std::thread> pool;
  int nslots = (int)P.devices.size();
  for (int w = 0; w < workers_per_device; w++)
    for (int s = 0; s < nslots; s++) {
      if (w == 0 && s == 0) continue;
      pool.emplace_back(work, s);
    }
  work(0);
  for (auto& t : pool) t.join();
  return first_rc.load();
}

// all-reduce (sum) of one integer across the group: a barrier that also spreads a failure flag
inline int32_t dist_sum(int32_t mine, int32_t* total, char* err, size_t errcap) {
  DistState& d = dist_state();
  *total = mine;
  if (!d.on || d.world == 1) return SSO_OK;
  const NcclApi* api = nccl_api(err, errcap);
  if (!api) return SSO_E_CUDA;
  Ctx c(err, errcap);
  int rc = c.init(d.device);
  if (rc) return rc;
  int32_t* d_v;
  if ((rc = c.alloc((void**)&d_v, 4))) return rc;
  CUDA_TRY(cudaMemcpyAsync(d_v, &mine, 4, cudaMemcpyHostToDevice, c.s[0]));
  {
    std::lock_guard<std::mutex> g(dist_mutex());
    NCCL_TRY(api, api->AllReduce(d_v, d_v, 1, ncclInt32, ncclSum, d.comm, c.s[0]));
  }
  CUDA_TRY(cudaMemcpyAsync(total, d_v, 4, cudaMemcpyDeviceToHost, c.s[0]));
  CUDA_TRY(cudaStreamSynchronize(c.s[0]));
  return SSO_OK;
}

// Every rank of a cooperative call must take the same path through the collectives: after a phase that can fail on one
// rank only (a bad element sits in ONE rank's piece), the failure flags are summed and every rank leaves together.
inline int32_t agree(const Participants& P, int32_t rc, char* err, size_t errcap) {
  if (!P.dist) return rc;
  int32_t total = 0;
  char e2[256];
  e2[0] = 0;
  int32_t rc2 = dist_sum(rc != SSO_OK ? 1 : 0, &total, e2, sizeof e2);
  if (rc != SSO_OK) return rc;
  if (rc2 != SSO_OK) { set_err(err, errcap, "%s", e2); return rc2; }
  if (total != 0) { set_err(err, errcap, "another rank of the process group rejected its share of the call"); return SSO_E_VERIFY; }
  return SSO_OK;
}

// ---------------------------------------------------------------------------------------------
// Decode / check / re-encode vectors in pieces, with optional power_pairs partial sums
// ---------------------------------------------------------------------------------------------
struct RVec {
  uint32_t group;
  const uint8_t* in; uint32_t in_compressed; uint64_t n;
  uint8_t* out; uint32_t out_compressed;          // out may be null (checks / pairs only)
  uint32_t want_pairs;                             // accumulate (sum r_i v_i, sum r_i v_{i+1})
  uint32_t check, subgroup;
  uint64_t tweak_id;                               // names the vector in the derivation of the MSM scalars
  const char* name;
};
struct RPiece { uint32_t vec; uint64_t lo, cnt; };  // elements [lo, lo + cnt); pairs [lo, lo + cnt - 1) when want_pairs

inline size_t point_size(const CurveSizes& cs, uint32_t group, uint32_t compressed) {
  return group == GROUP_G1 ? (compressed ? cs.g1c : cs.g1u) : (compressed ? cs.g2c : cs.g2u);
}
inline void identity_bytes(uint8_t* dst, size_t usz) { memset(dst, 0, usz); dst[usz - 1] = 0x40; }

// Sum of `cnt` uncompressed points held on the host, computed on the context's device; cnt == 0 gives the identity.
inline int sum_points_host(Ctx& c, const CurveOps* ops, uint32_t group, size_t usz, const uint8_t* pts, size_t cnt, uint8_t* out,
                           char* err, size_t errcap) {
  if (cnt == 0) { identity_bytes(out, usz); return SSO_OK; }
  if (cnt == 1) { memcpy(out, pts, usz); return SSO_OK; }
  uint8_t *d_in, *d_out;
  uint32_t* d_status;
  int rc;
  if ((rc = c.alloc((void**)&d_in, cnt * usz))) return rc;
  if ((rc = c.alloc((void**)&d_out, usz))) return rc;
  if ((rc = status_buffer(c, &d_status, 0, false, err, errcap))) return rc;
  CUDA_TRY(cudaMemcpyAsync(d_in, pts, cnt * usz, cudaMemcpyHostToDevice, c.s[0]));
  if ((rc = ops->points_sum(c, 0, group, d_in, (uint32_t)cnt, d_out, d_status, err, errcap))) return rc;
  CUDA_TRY(cudaMemcpyAsync(out, d_out, usz, cudaMemcpyDeviceToHost, c.s[0]));
  CUDA_TRY(cudaStreamSynchronize(c.s[0]));
  return check_status(c, d_status, "partial sum", err, errcap);
}

// All-gather of one blob per participant (device-resident on each participant's device) and the sums that follow.
//   mine[slot]  : host copy of participant `slot`'s blob (nvec pairs: A | B per vector, uncompressed)
// Returns the summed pairs (host) in `pairs`.  One participant: no collective.
inline int exchange_and_sum(const CurveOps* ops, const CurveSizes& cs, const Participants& P, const std::vector<RVec>& vecs,
                            const std::vector<std::vector<uint8_t>>& mine, std::vector<std::vector<uint8_t>>& pairs, char* err, size_t errcap) {
  const size_t nvec = vecs.size();
  size_t blob = 0;
  std::vector<size_t> voff(nvec), vusz(nvec);
  for (size_t v = 0; v < nvec; v++) { vusz[v] = point_size(cs, vecs[v].group, 0); voff[v] = blob; blob += 2 * vusz[v]; }
  const int nlocal = (int)P.devices.size();
  const int total = P.dist ? P.world : nlocal;
  pairs.assign(nvec, {});
  if (total == 1) {
    for (size_t v = 0; v < nvec; v++) pairs[v].assign(mine[0].begin() + voff[v], mine[0].begin() + voff[v] + 2 * vusz[v]);
    return SSO_OK;
  }
  const NcclApi* api = nccl_api(err, errcap);
  if (!api) return SSO_E_CUDA;
  // device buffers: send (blob) and receive (total * blob) on every local participant
  std::vector<std::unique_ptr<Ctx>> ctx(nlocal);
  std::vector<uint8_t*> d_send(nlocal), d_recv(nlocal);
  std::vector<ncclComm_t> comms(nlocal);
  int rc;
  if (P.dist) comms[0] = dist_state().comm;
  else {
    LocalComms* lc;
    if ((rc = local_comms(P.devices, &lc, err, errcap))) return rc;
    comms = lc->comms;
  }
  for (int s = 0; s < nlocal; s++) {
    ctx[s].reset(new Ctx(err, errcap));
    if ((rc = ctx[s]->init(P.devices[s]))) return rc;
    if ((rc = ctx[s]->alloc((void**)&d_send[s], blob))) return rc;
    if ((rc = ctx[s]->alloc((void**)&d_recv[s], blob * total))) return rc;
    CUDA_TRY(cudaMemcpyAsync(d_send[s], mine[s].data(), blob, cudaMemcpyHostToDevice, ctx[s]->s[0]));
  }
  {
    std::lock_guard<std::mutex> g(dist_mutex());           // one collective at a time per process
    NCCL_TRY(api, api->GroupStart());
    for (int s = 0; s < nlocal; s++) {
      CUDA_TRY(cudaSetDevice(P.devices[s]));
      NCCL_TRY(api, api->AllGather(d_send[s], d_recv[s], blob, ncclUint8, comms[s], ctx[s]->s[0]));
    }
    NCCL_TRY(api, api->GroupEnd());
    dist_state().collectives++;
  }
  for (int s = 0; s < nlocal; s++) { CUDA_TRY(cudaSetDevice(P.devices[s])); CUDA_TRY(cudaStreamSynchronize(ctx[s]->s[0])); }
  // the point addition that follows the gather: participant 0 of this process sums the `total` partial points of every slot
  Ctx& c = *ctx[0];
  CUDA_TRY(cudaSetDevice(P.devices[0]));
  for (size_t v = 0; v < nvec; v++) {
    pairs[v].resize(2 * vusz[v]);
    for (int half = 0; half < 2; half++) {
      uint8_t *d_pts, *d_out;
      uint32_t* d_status;
      if ((rc = c.alloc((void**)&d_pts, vusz[v] * total))) return rc;
      if ((rc = c.alloc((void**)&d_out, vusz[v]))) return rc;
      if ((rc = status_buffer(c, &d_status, 0, false, err, errcap))) return rc;
      CUDA_TRY(cudaMemcpy2DAsync(d_pts, vusz[v], d_recv[0] + voff[v] + half * vusz[v], blob, vusz[v], total, cudaMemcpyDeviceToDevice, c.s[0]));
      if ((rc = ops->points_sum(c, 0, vecs[v].group, d_pts, (uint32_t)total, d_out, d_status, err, errcap))) return rc;
      CUDA_TRY(cudaMemcpyAsync(pairs[v].data() + half * vusz[v], d_out, vusz[v], cudaMemcpyDeviceToHost, c.s[0]));
      CUDA_TRY(cudaStreamSynchronize(c.s[0]));
      if ((rc = check_status(c, d_status, "gathered partial point", err, errcap))) return rc;
    }
  }
  return SSO_OK;
}

// The engine.  pairs[v] (2 uncompressed points) is filled for vectors with want_pairs (identity pair when n < 2).
inline int stream_reencode(const CurveOps* ops, const CurveSizes& cs, const std::vector<RVec>& vecs, uint64_t piece_elems,
                           const uint8_t* rlc_seed32, uint64_t tweak_chunk, const Participants& P,
                           std::vector<std::vector<uint8_t>>* pairs, char* err, size_t errcap) {
  if (piece_elems == 0) piece_elems = 1ull << 20;
  if (piece_elems > (1ull << 22)) piece_elems = 1ull << 22;
  std::vector<RPiece> pieces;
  bool any_pairs = false;
  for (size_t v = 0; v < vecs.size(); v++) {
    const RVec& r = vecs[v];
    if (r.n == 0) continue;
    if (r.want_pairs && r.n >= 2) {
      any_pairs = true;
      for (uint64_t lo = 0; lo < r.n - 1; lo += piece_elems) {
        uint64_t hi = lo + piece_elems < r.n - 1 ? lo + piece_elems : r.n - 1;
        pieces.push_back({(uint32_t)v, lo, hi - lo + 1});
      }
    } else {
      for (uint64_t lo = 0; lo < r.n; lo += piece_elems) pieces.push_back({(uint32_t)v, lo, lo + piece_elems < r.n ? piece_elems : r.n - lo});
    }
  }
  const int nlocal = (int)P.devices.size();
  // partial pairs per local participant and vector
  std::vector<std::vector<std::vector<uint8_t>>> part(nlocal, std::vector<std::vector<uint8_t>>(vecs.size()));
  std::mutex part_lock;
  int rc = run_pieces(pieces.size(), P, 2, 1, err, errcap, [&](size_t i, int slot, Ctx& c, char* e, size_t ec) -> int {
    char* err = e; size_t errcap = ec;            // CUDA_TRY reports into the worker's buffer
    const RPiece& pc = pieces[i];
    const RVec& r = vecs[pc.vec];
    const size_t isz = point_size(cs, r.group, r.in_compressed), osz = point_size(cs, r.group, r.out_compressed), usz = point_size(cs, r.group, 0);
    const bool pairs_here = r.want_pairs && pc.cnt >= 2;
    uint8_t *d_in, *d_out = nullptr, *d_pair = nullptr;
    uint32_t *d_aff = nullptr, *d_status;
    int rc;
    if ((rc = c.alloc((void**)&d_in, pc.cnt * isz))) return rc;
    if (r.out && (rc = c.alloc((void**)&d_out, pc.cnt * osz))) return rc;
    if (pairs_here && (rc = c.alloc((void**)&d_aff, pc.cnt * ops->aff_words[r.group] * 4))) return rc;
    if (pairs_here && (rc = c.alloc((void**)&d_pair, 2 * usz))) return rc;
    if ((rc = status_buffer(c, &d_status, 0, false, err, errcap))) return rc;
    CUDA_TRY(cudaMemcpyAsync(d_in, r.in + pc.lo * isz, pc.cnt * isz, cudaMemcpyHostToDevice, c.s[0]));
    if ((rc = ops->reencode(c, 0, r.group, d_in, r.in_compressed, pc.cnt, d_out, r.out_compressed, r.check, r.subgroup, d_aff, d_status, e, ec))) return rc;
    std::vector<uint8_t> pair;
    if (pairs_here) {
      const uint64_t tweak[4] = {r.tweak_id, tweak_chunk, pc.lo, (uint64_t)P.rank * 64 + (uint64_t)slot};
      if ((rc = ops->msm_pairs(c, 0, r.group, d_aff, d_aff + ops->aff_words[r.group], pc.cnt - 1, rlc_seed32, tweak, d_pair, e, ec))) return rc;
      pair.resize(2 * usz);
      CUDA_TRY(cudaMemcpyAsync(pair.data(), d_pair, 2 * usz, cudaMemcpyDeviceToHost, c.s[0]));
    }
    if (r.out) CUDA_TRY(cudaMemcpyAsync(r.out + pc.lo * osz, d_out, pc.cnt * osz, cudaMemcpyDeviceToHost, c.s[0]));
    CUDA_TRY(cudaStreamSynchronize(c.s[0]));
    uint32_t h[4] = {0, 0, 0, 0};
    CUDA_TRY(cudaMemcpy(h, d_status, STATUS_BYTES, cudaMemcpyDeviceToHost));
    if (h[0] != 0) {
      set_err(e, ec, "%s: %s (element %llu)", r.name ? r.name : "vector", status_text(h[0]), (unsigned long long)(pc.lo + h[1]));
      return h[0] == 5u ? SSO_E_VERIFY : SSO_E_INPUT;
    }
    if (pairs_here) {
      std::lock_guard<std::mutex> g(part_lock);
      auto& dst = part[slot][pc.vec];
      dst.insert(dst.end(), pair.begin(), pair.end());
    }
    return SSO_OK;
  });
  if ((rc = agree(P, rc, err, errcap))) return rc;
  if (!pairs) return SSO_OK;
  if (!any_pairs) {
    pairs->assign(vecs.size(), {});
    for (size_t v = 0; v < vecs.size(); v++) {
      size_t usz = point_size(cs, vecs[v].group, 0);
      (*pairs)[v].resize(2 * usz);
      identity_bytes((*pairs)[v].data(), usz);
      identity_bytes((*pairs)[v].data() + usz, usz);
    }
    return SSO_OK;
  }
  // per participant: fold its pieces' partial pairs on its own device
  size_t blob = 0;
  std::vector<size_t> voff(vecs.size()), vusz(vecs.size());
  for (size_t v = 0; v < vecs.size(); v++) { vusz[v] = point_size(cs, vecs[v].group, 0); voff[v] = blob; blob += 2 * vusz[v]; }
  std::vector<std::vector<uint8_t>> mine(nlocal, std::vector<uint8_t>(blob));
  auto fold = [&]() -> int {
    int rc;
    for (int s = 0; s < nlocal; s++) {
      Ctx c(err, errcap);
      if ((rc = c.init(P.devices[s]))) return rc;
      for (size_t v = 0; v < vecs.size(); v++) {
        const size_t usz = vusz[v], cnt = part[s][v].size() / (2 * usz);
        std::vector<uint8_t> a(cnt * usz), b(cnt * usz);
        for (size_t k = 0; k < cnt; k++) {
          memcpy(a.data() + k * usz, part[s][v].data() + k * 2 * usz, usz);
          memcpy(b.data() + k * usz, part[s][v].data() + k * 2 * usz + usz, usz);
        }
        if ((rc = sum_points_host(c, ops, vecs[v].group, usz, a.data(), cnt, mine[s].data() + voff[v], err, errcap))) return rc;
        if ((rc = sum_points_host(c, ops, vecs[v].group, usz, b.data(), cnt, mine[s].data() + voff[v] + usz, err, errcap))) return rc;
      }
    }
    return SSO_OK;
  };
  if ((rc = agree(P, fold(), err, errcap))) return rc;
  return exchange_and_sum(ops, cs, P, vecs, mine, *pairs, err, errcap);
}

// ---------------------------------------------------------------------------------------------
// Phase1::computation in pieces: challenge (uncompressed, host) -> response vectors (compressed, host).
// Coefficient slots as in p1_contribute_streams: tauG1 / tauG2 plain powers, alphaG1 * alpha, betaG1 * beta, betaG2 = beta.
// ---------------------------------------------------------------------------------------------
inline int stream_contribute(const CurveOps* ops, const P1Layout& L, const uint8_t* challenge, uint8_t* response, const uint8_t* tau,
                             const uint8_t* alpha, const uint8_t* beta, uint32_t check, uint64_t piece_elems, const Participants& P,
                             char* err, size_t errcap) {
  if (piece_elems == 0) piece_elems = 1ull << 20;
  if (piece_elems > (1ull << 22)) piece_elems = 1ull << 22;
  struct CPiece { uint32_t vec; uint64_t lo, cnt; };
  std::vector<CPiece> pieces;
  const uint64_t counts[5] = {L.g1n, L.on, L.on, L.on, 1};
  static const uint32_t groups[5] = {GROUP_G1, GROUP_G2, GROUP_G1, GROUP_G1, GROUP_G2};
  static const uint32_t slot[5] = {0, 0, 1, 2, 2}, has_coeff[5] = {0, 0, 1, 1, 1}, mode[5] = {0, 0, 0, 0, 1};
  // G2 pieces first: they run longest, the G1 pieces fill the tail of the queue
  const int order[5] = {1, 4, 0, 2, 3};
  for (int oi = 0; oi < 5; oi++) {
    int v = order[oi];
    for (uint64_t lo = 0; lo < counts[v]; lo += piece_elems) pieces.push_back({(uint32_t)v, lo, lo + piece_elems < counts[v] ? piece_elems : counts[v] - lo});
  }
  int rc_all = run_pieces(pieces.size(), P, 2, 1, err, errcap, [&](size_t i, int, Ctx& c, char* e, size_t ec) -> int {
    char* err = e; size_t errcap = ec;
    const CPiece& pc = pieces[i];
    const uint32_t g = groups[pc.vec];
    const size_t usz = point_size(L.cs, g, 0), csz = point_size(L.cs, g, 1);
    uint8_t *d_in, *d_out;
    uint32_t *d_status, *d_table;
    int rc;
    if ((rc = c.alloc((void**)&d_in, pc.cnt * usz))) return rc;
    if ((rc = c.alloc((void**)&d_out, pc.cnt * csz))) return rc;
    if ((rc = status_buffer(c, &d_status, 0, false, err, errcap))) return rc;
    CUDA_TRY(cudaMemcpyAsync(d_in, challenge + L.off_u[pc.vec] + pc.lo * usz, pc.cnt * usz, cudaMemcpyHostToDevice, c.s[0]));
    if (check == CHECK_FULL) {                     // CheckForCorrectness::Full on the inputs: on the curve AND in the subgroup
      if ((rc = ops->reencode(c, 0, g, d_in, 0, pc.cnt, nullptr, 0, CHECK_FULL, 1, nullptr, d_status, e, ec))) return rc;
    }
    const uint8_t* coeffs[TAU_COEFF_SLOTS] = {nullptr, alpha, beta};
    if ((rc = ops->tau_tables(c, 0, L.start + pc.lo, tau, coeffs, &d_table, e, ec))) return rc;
    VecBatch b;
    memset(&b, 0, sizeof b);
    b.seg[0].in = d_in; b.seg[0].out = d_out; b.seg[0].n = (uint32_t)pc.cnt; b.seg[0].coeff_slot = slot[pc.vec];
    b.seg[0].has_coeff = has_coeff[pc.vec]; b.seg[0].mode = mode[pc.vec];
    b.nseg = 1; b.total = (uint32_t)pc.cnt;
    if ((rc = ops->batch_exp(c, 0, g, b, 0, d_table, 1, check, d_status, e, ec))) return rc;
    CUDA_TRY(cudaMemcpyAsync(response + L.off_c[pc.vec] + pc.lo * csz, d_out, pc.cnt * csz, cudaMemcpyDeviceToHost, c.s[0]));
    CUDA_TRY(cudaStreamSynchronize(c.s[0]));
    uint32_t h[4] = {0, 0, 0, 0};
    CUDA_TRY(cudaMemcpy(h, d_status, STATUS_BYTES, cudaMemcpyDeviceToHost));
    if (h[0] != 0) {
      set_err(e, ec, "challenge: %s (vector %u, element %llu)", status_text(h[0]), pc.vec, (unsigned long long)(pc.lo + h[1]));
      return h[0] == 5u ? SSO_E_VERIFY : SSO_E_INPUT;
    }
    return SSO_OK;
  });
  return agree(P, rc_all, err, errcap);
}

}  // namespace sso
