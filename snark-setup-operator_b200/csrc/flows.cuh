// Host-side orchestration of the file-level ceremony calls (SURVEY.md §8a rows a2, a3, a5, a12, a13):
// what phase1_cli::contribute and phase1_cli::transform_pok_and_correctness do around the kernels —
// size asserts, the Blake2b hash chain, key generation from the seeded RNG, the proof-of-knowledge and
// ratio checks — expressed over the CurveOps table.  All arithmetic runs on the device.
#pragma once
#include <thread>
#include <mutex>
#include <atomic>

#include "blake2b.h"
#include "curve_ops.cuh"
#include "stream.cuh"

namespace sso {

// joins the thread when the scope ends, on an early return too
struct JoinOnExit {
  std::thread& t;
  ~JoinOnExit() { if (t.joinable()) t.join(); }
};

// ---- key generation (Phase1::key_generation) ---------------------------------------------------
// seed32: ChaCha20 seed of the contributor RNG; digest64: Blake2b(challenge).
// scalars_out: nscalars canonical scalars (fr_bytes each); pubkey_out: 2*nscalars G1 + nscalars G2 uncompressed.
// Key generation in two stages so that the digest-independent half can run before the challenge hash is known:
//   stage 1 (seed only)   : the private scalars and the (s, s^x) G1 pairs of the proofs of knowledge — the RNG draws
//   stage 2 (needs digest): compute_g2_s = hash_to_g2(Blake2b(personalization || digest || g1_s || g1_s_x)[..32]) and
//                           its multiple by the scalar; the public key is the G1 pairs followed by the G2 points
struct KeygenState {
  uint32_t nscalars = 0;
  uint32_t *d_scalars = nullptr, *d_seeds2 = nullptr;
  uint8_t *d_g2s = nullptr, *d_g2sx = nullptr, *d_g1 = nullptr;
  std::vector<uint8_t> g1, seeds2;
  std::vector<uint32_t> sc;
};
inline int keygen_stage1(Ctx& c, int si, const CurveOps* ops, const CurveSizes& cs, const uint8_t seed32[32], uint32_t nscalars,
                         KeygenState& k, uint8_t* scalars_out, char* err, size_t errcap) {
  int rc;
  uint32_t* d_seed;
  uint8_t* d_g1;
  const size_t g1u = cs.g1u, g2u = cs.g2u;
  k.nscalars = nscalars;
  if ((rc = c.alloc((void**)&d_seed, 32, si))) return rc;
  if ((rc = c.alloc((void**)&k.d_scalars, (size_t)nscalars * ops->fr_words * 4, si))) return rc;
  if ((rc = c.alloc((void**)&d_g1, 2 * nscalars * g1u, si))) return rc;
  if ((rc = c.alloc((void**)&k.d_seeds2, (size_t)nscalars * 32, si))) return rc;
  if ((rc = c.alloc((void**)&k.d_g2s, nscalars * g2u, si))) return rc;
  if ((rc = c.alloc((void**)&k.d_g2sx, nscalars * g2u, si))) return rc;
  CUDA_TRY(cudaMemcpyAsync(d_seed, seed32, 32, cudaMemcpyHostToDevice, c.s[si]));
  // the scalars first (microseconds): the caller starts its main kernels with them; the point sampling and the G1 halves of
  // the proofs (a single-thread kernel of ~20 ms) stay enqueued on this stream and are collected by stage 2
  uint32_t* d_sc_only;
  if ((rc = c.alloc((void**)&d_sc_only, (size_t)nscalars * ops->fr_words * 4, si))) return rc;
  if ((rc = ops->keygen_scalars(c, si, d_seed, nscalars, d_sc_only, err, errcap))) return rc;
  k.sc.resize((size_t)nscalars * ops->fr_words);
  CUDA_TRY(cudaMemcpyAsync(k.sc.data(), d_sc_only, k.sc.size() * 4, cudaMemcpyDeviceToHost, c.s[si]));
  CUDA_TRY(cudaStreamSynchronize(c.s[si]));
  for (uint32_t i = 0; i < nscalars; i++)
    memcpy(scalars_out + (size_t)i * ops->fr_bytes, k.sc.data() + (size_t)i * ops->fr_words, ops->fr_bytes);
  if ((rc = ops->keygen_g1(c, si, d_seed, nscalars, k.d_scalars, d_g1, err, errcap))) return rc;
  k.d_g1 = d_g1;
  return SSO_OK;
}
// waits for the G1 halves of the proofs left running by stage 1: k.g1 = g1_s(x) | g1_s_x(x) per scalar, uncompressed
inline int keygen_collect_g1(Ctx& c, int si, const CurveSizes& cs, KeygenState& k, char* err, size_t errcap) {
  if (!k.g1.empty()) return SSO_OK;
  k.g1.resize(2 * k.nscalars * cs.g1u);
  CUDA_TRY(cudaMemcpyAsync(k.g1.data(), k.d_g1, k.g1.size(), cudaMemcpyDeviceToHost, c.s[si]));
  CUDA_TRY(cudaStreamSynchronize(c.s[si]));
  return SSO_OK;
}
// enqueues on stream si (the stream stage 1 ran on); pubkey_out is complete once si drained
inline int keygen_stage2(Ctx& c, int si, const CurveOps* ops, const CurveSizes& cs, const uint8_t digest64[64], KeygenState& k,
                         uint8_t* pubkey_out, char* err, size_t errcap) {
  int rc;
  const size_t g1u = cs.g1u, g2u = cs.g2u;
  if ((rc = keygen_collect_g1(c, si, cs, k, err, errcap))) return rc;
  // compute_g2_s: Blake2b(personalization || digest || g1_s || g1_s_x)[..32] seeds hash_to_g2
  k.seeds2.resize((size_t)k.nscalars * 32);
  for (uint32_t i = 0; i < k.nscalars; i++) {
    Blake2b h(64);
    uint8_t pers = (uint8_t)i, full[64];
    h.update(&pers, 1);
    h.update(digest64, 64);
    h.update(k.g1.data() + (size_t)2 * i * g1u, 2 * g1u);
    h.final(full, 64);
    memcpy(k.seeds2.data() + 32 * i, full, 32);
  }
  CUDA_TRY(cudaMemcpyAsync(k.d_seeds2, k.seeds2.data(), k.seeds2.size(), cudaMemcpyHostToDevice, c.s[si]));
  if ((rc = ops->hash_to_g2(c, si, k.nscalars, k.d_seeds2, k.d_scalars, k.d_g2s, k.d_g2sx, err, errcap))) return rc;
  memcpy(pubkey_out, k.g1.data(), k.g1.size());
  CUDA_TRY(cudaMemcpyAsync(pubkey_out + k.g1.size(), k.d_g2sx, k.nscalars * g2u, cudaMemcpyDeviceToHost, c.s[si]));
  return SSO_OK;
}
inline int keygen_host(Ctx& c, const CurveOps* ops, const CurveSizes& cs, const uint8_t seed32[32], const uint8_t digest64[64],
                       uint32_t nscalars, uint8_t* scalars_out, uint8_t* pubkey_out, char* err, size_t errcap) {
  KeygenState k;
  int rc;
  if ((rc = keygen_stage1(c, 0, ops, cs, seed32, nscalars, k, scalars_out, err, errcap))) return rc;
  if ((rc = keygen_stage2(c, 0, ops, cs, digest64, k, pubkey_out, err, errcap))) return rc;
  CUDA_TRY(cudaStreamSynchronize(c.s[0]));
  return SSO_OK;
}

// ---- generators -------------------------------------------------------------------------------------
// The G1 / G2 generators new_challenge writes and chunk-0 verification compares against.  The built-in constants are
// arkworks' for BLS12-377, BW6-761 and both G1 of the MNT curves; the G2 generators of MNT4-753 / MNT6-753 could not be
// recovered in this environment (DESIGN.md §2) and default to a derived order-r point, so the host application hands the
// reference's constants over once per process (sso_p1_set_generators) — e.g. read from the round-0 challenge the
// operator regenerates and compares by hash (reference src/bin/verify_transcript.rs:316-361).
struct GenOverride { bool set = false; std::vector<uint8_t> g1u, g2u; };
inline GenOverride& gen_override(uint32_t curve) { static GenOverride g[4]; return g[curve & 3]; }
inline std::mutex& gen_mutex() { static std::mutex m; return m; }

// uncompressed generator bytes (g1u | g2u) into `out`
inline int generator_bytes(Ctx& c, const CurveOps* ops, const CurveSizes& cs, uint32_t curve, uint8_t* out, char* err, size_t errcap) {
  {
    std::lock_guard<std::mutex> g(gen_mutex());
    const GenOverride& o = gen_override(curve);
    if (o.set) { memcpy(out, o.g1u.data(), cs.g1u); memcpy(out + cs.g1u, o.g2u.data(), cs.g2u); return SSO_OK; }
  }
  uint8_t* d_gen;
  int rc;
  if ((rc = c.alloc((void**)&d_gen, cs.g1u + cs.g2u))) return rc;
  if ((rc = ops->fill_generator(c, 0, GROUP_G1, 1, d_gen, 0, err, errcap))) return rc;
  if ((rc = ops->fill_generator(c, 0, GROUP_G2, 1, d_gen + cs.g1u, 0, err, errcap))) return rc;
  CUDA_TRY(cudaMemcpyAsync(out, d_gen, cs.g1u + cs.g2u, cudaMemcpyDeviceToHost, c.s[0]));
  CUDA_TRY(cudaStreamSynchronize(c.s[0]));
  return SSO_OK;
}

// ---- chunk verification (Phase1::verification) ----------------------------------------------------------
struct RatioCheck { std::string name; std::vector<uint8_t> bytes; };

inline void add_check(std::vector<RatioCheck>& v, const char* name, const uint8_t* a, const uint8_t* b, size_t g1u, const uint8_t* cc,
                      const uint8_t* d, size_t g2u) {
  RatioCheck r;
  r.name = name;
  r.bytes.resize(2 * g1u + 2 * g2u);
  memcpy(r.bytes.data(), a, g1u);
  memcpy(r.bytes.data() + g1u, b, g1u);
  memcpy(r.bytes.data() + 2 * g1u, cc, g2u);
  memcpy(r.bytes.data() + 2 * g1u + g2u, d, g2u);
  v.push_back(std::move(r));
}

// runs all collected same_ratio checks in one launch; SSO_E_VERIFY names the first failing one
inline int run_checks(Ctx& c, const CurveOps* ops, const std::vector<RatioCheck>& checks, char* err, size_t errcap) {
  if (checks.empty()) return SSO_OK;
  size_t cb = ops->check_bytes, n = checks.size();
  std::vector<uint8_t> flat(n * cb);
  for (size_t i = 0; i < n; i++) memcpy(flat.data() + i * cb, checks[i].bytes.data(), cb);
  uint8_t* d_checks;
  uint32_t* d_verdicts;
  int rc;
  if ((rc = c.alloc((void**)&d_checks, flat.size()))) return rc;
  if ((rc = c.alloc((void**)&d_verdicts, n * 4))) return rc;
  CUDA_TRY(cudaMemcpyAsync(d_checks, flat.data(), flat.size(), cudaMemcpyHostToDevice, c.s[0]));
  if ((rc = ops->same_ratio(c, 0, d_checks, n, d_verdicts, err, errcap))) return rc;
  std::vector<uint32_t> v(n);
  CUDA_TRY(cudaMemcpyAsync(v.data(), d_verdicts, n * 4, cudaMemcpyDeviceToHost, c.s[0]));
  CUDA_TRY(cudaStreamSynchronize(c.s[0]));
  for (size_t i = 0; i < n; i++) {
    if (v[i] >= 0x100u) { set_err(err, errcap, "same_ratio check '%s': %s", checks[i].name.c_str(), status_text(v[i] - 0x100u)); return SSO_E_VERIFY; }
    if (v[i] != 1u) { set_err(err, errcap, "same_ratio check failed: %s", checks[i].name.c_str()); return SSO_E_VERIFY; }
  }
  return SSO_OK;
}

// The per-element policy of the verification (SURVEY.md §8a rows a5, a14; reference src/bin/contribute.rs:966-987):
//   every response element must be non-zero, whatever `check_output` says ([UP] Phase1::verification reads the batches
//   with OnlyNonZero); CheckForCorrectness::Full adds nothing for compressed input (decompression lands on the curve)
//   but, being the "force correctness checks" setting, also forces the membership test;
//   SubgroupCheckMode::{Auto, Direct, Batched} ask for the membership test, ::No skips it.
inline uint32_t verify_elem_check(uint32_t check_output) { return check_output == CHECK_NO ? (uint32_t)CHECK_NONZERO : check_output; }
inline uint32_t verify_subgroup(uint32_t check_output, uint32_t subgroup_mode) {
  return (subgroup_mode != SSO_SUBGROUP_NO || check_output == CHECK_FULL) ? 1u : 0u;
}
// tweak words naming the MSMs of one verification (curve_ops.cuh::run_msm_pairs)
static constexpr uint64_t TWEAK_P1_VERIFY = 0x7031760000000000ull, TWEAK_P1_RATIOS = 0x7031720000000000ull, TWEAK_P2_VERIFY = 0x7032760000000000ull;

// challenge (uncompressed, host) + response (compressed + pubkey, host) -> new_challenge (uncompressed, host).
//   P == nullptr : the chunk is resident on the context's device (two streams, all vectors at once)
//   P != nullptr : vectors streamed in pieces of `piece_elems` over the participants (Full mode / large chunks)
// rlc_seed32: NULL = fresh entropy for the random linear combinations (the only sound setting outside tests).
inline int verify_chunk_host(Ctx& c, const CurveOps* ops, const P1Layout& L, uint32_t curve, uint64_t chunk_index,
                             const uint8_t* challenge, const uint8_t* response, uint8_t* new_challenge, uint32_t check_input,
                             uint32_t check_output, uint32_t subgroup_mode, uint32_t ratio_check, const uint8_t* rlc_seed32,
                             const Participants* P, uint64_t piece_elems, uint8_t* ch_hash_out, char* err, size_t errcap) {
  int rc;
  const size_t g1u = L.cs.g1u, g2u = L.cs.g2u;
  const uint64_t counts[5] = {L.g1n, L.on, L.on, L.on, 1};
  static const uint32_t groups[5] = {GROUP_G1, GROUP_G2, GROUP_G1, GROUP_G1, GROUP_G2};
  static const char* vnames[5] = {"response tau_g1", "response tau_g2", "response alpha_g1", "response beta_g1", "response beta_g2"};
  static const char* inames[5] = {"challenge tau_g1", "challenge tau_g2", "challenge alpha_g1", "challenge beta_g1", "challenge beta_g2"};
  const uint32_t elem_check = verify_elem_check(check_output), subgroup = verify_subgroup(check_output, subgroup_mode);
  // Beside the main GPU work, on a host thread with its own high-priority stream: Blake2b(challenge) (sequential, the longest
  // host step), then — the digest known — the public-key validation and g2_s = hash_to_g2(Blake2b(pers || digest || g1_s ||
  // g1_s_x)) of the three proofs (single-thread chains of tens of milliseconds that would otherwise run after everything
  // else), and Blake2b(response) while those kernels run.
  struct Side { int rc = SSO_OK; char err[256]; uint8_t ch_hash[64], resp_hash[64]; std::vector<uint8_t> g2s; } side;
  side.err[0] = 0;
  const uint8_t* pk = response + L.off_c[5];
  const int side_device = c.dev;
  // the response hash has its own thread: at accumulator scale (a gigabyte and more) the two sequential Blake2b passes are
  // the critical path of the call (~1 GB/s each)
  std::thread resp_hasher([&] { blake2b_512(response, L.contrib_size, side.resp_hash); });
  JoinOnExit join_resp_hasher{resp_hasher};
  std::thread side_thread([&] {
    char* err = side.err; size_t errcap = sizeof side.err;
    side.rc = [&]() -> int {
      int rc;
      blake2b_512(challenge, L.acc_size, side.ch_hash);
      Ctx c2(err, errcap);
      if ((rc = c2.init(side_device, 3))) return rc;
      const int si = c2.aliased ? 0 : 2;
      // the public key: nine points that must be non-zero, on their curves and in the subgroups (a zero or torsion point
      // would make the proof-of-knowledge pairings vacuous)
      uint8_t *d_pk, *d_g2s;
      uint32_t *d_status, *d_seeds2;
      if ((rc = c2.alloc((void**)&d_pk, L.pk_size, si))) return rc;
      if ((rc = status_buffer(c2, &d_status, si, false, err, errcap))) return rc;
      if ((rc = c2.alloc((void**)&d_seeds2, 96, si))) return rc;
      if ((rc = c2.alloc((void**)&d_g2s, 3 * g2u, si))) return rc;
      CUDA_TRY(cudaMemcpyAsync(d_pk, pk, L.pk_size, cudaMemcpyHostToDevice, c2.s[si]));
      if ((rc = ops->reencode(c2, si, GROUP_G1, d_pk, 0, 6, nullptr, 0, CHECK_FULL, 1, nullptr, d_status, err, errcap))) return rc;
      if ((rc = ops->reencode(c2, si, GROUP_G2, d_pk + 6 * g1u, 0, 3, nullptr, 0, CHECK_FULL, 1, nullptr, d_status, err, errcap))) return rc;
      std::vector<uint8_t> seeds2(3 * 32);
      for (uint32_t i = 0; i < 3; i++) {
        Blake2b h(64);
        uint8_t pers = (uint8_t)i, full[64];
        h.update(&pers, 1);
        h.update(side.ch_hash, 64);
        h.update(pk + (size_t)2 * i * g1u, 2 * g1u);
        h.final(full, 64);
        memcpy(seeds2.data() + 32 * i, full, 32);
      }
      CUDA_TRY(cudaMemcpyAsync(d_seeds2, seeds2.data(), 96, cudaMemcpyHostToDevice, c2.s[si]));
      if ((rc = ops->hash_to_g2(c2, si, 3, d_seeds2, nullptr, d_g2s, nullptr, err, errcap))) return rc;
      side.g2s.resize(3 * g2u);
      CUDA_TRY(cudaMemcpyAsync(side.g2s.data(), d_g2s, side.g2s.size(), cudaMemcpyDeviceToHost, c2.s[si]));
      CUDA_TRY(cudaStreamSynchronize(c2.s[si]));
      if ((rc = check_status(c2, d_status, "public key", err, errcap))) return rc == SSO_E_INPUT ? SSO_E_VERIFY : rc;
      return SSO_OK;
    }();
  });
  JoinOnExit join_side_thread{side_thread};
  std::vector<uint8_t> pairs[4];
  if (!P) {
    // 1. decode + check the response vectors on the device, producing the new challenge image
    uint8_t *d_resp, *d_new;
    uint32_t* d_status;
    if ((rc = c.alloc((void**)&d_resp, L.contrib_size))) return rc;
    if ((rc = c.alloc((void**)&d_new, L.acc_size))) return rc;
    if ((rc = status_buffer(c, &d_status, 0, false, err, errcap))) return rc;
    CUDA_TRY(cudaMemcpyAsync(d_resp, response, L.contrib_size, cudaMemcpyHostToDevice, c.s[0]));
    CUDA_TRY(cudaStreamSynchronize(c.s[0]));
    uint32_t* d_aff[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    if ((rc = c.fork(0, 1))) return rc;
    // the vectors go to the two streams by estimated device time, longest first onto the less loaded stream (on BLS12-377
    // that is tau_g2 + beta_g1 | tau_g1 + alpha_g1 instead of G2 | all of G1: the few-thread tails of one MSM then overlap
    // the other stream's work)
    int stream_of[5] = {0, 0, 0, 0, 0};
    {
      double cost[5], load[2] = {0.0, 0.0};
      int order[5] = {0, 1, 2, 3, 4};
      for (int v = 0; v < 5; v++) cost[v] = (double)counts[v] * (groups[v] == GROUP_G2 ? (double)ops->verify_g2_weight : 1.0);
      std::sort(order, order + 5, [&](int a, int b) { return cost[a] > cost[b]; });
      for (int k = 0; k < 5; k++) {
        int v = order[k], s = load[1] < load[0] ? 1 : 0;
        if (c.aliased) s = 0;
        stream_of[v] = s;
        load[s] += cost[v];
      }
    }
    for (int v = 0; v < 5; v++) {
      if (counts[v] == 0) continue;
      int si = stream_of[v];
      if (ratio_check && v < 4 && counts[v] >= 2)
        if ((rc = c.alloc((void**)&d_aff[v], counts[v] * ops->aff_words[groups[v]] * 4, si))) return rc;
      if ((rc = ops->reencode(c, si, groups[v], d_resp + L.off_c[v], 1, counts[v], d_new + L.off_u[v], 0, elem_check, subgroup,
                              d_aff[v], d_status, err, errcap))) return rc;
    }
    c.mark("verify: decode launches enqueued");
    // 2. random-linear-combination pairs for the power-ratio checks (every MSM with its own scalars)
    uint8_t* d_pairs[4] = {nullptr, nullptr, nullptr, nullptr};
    for (int v = 0; v < 4; v++) {
      if (!d_aff[v]) continue;
      int si = stream_of[v];
      const size_t usz = point_size(L.cs, groups[v], 0);
      const uint64_t tweak[4] = {TWEAK_P1_VERIFY | (uint64_t)v, chunk_index, 0, 0};
      if ((rc = c.alloc((void**)&d_pairs[v], 2 * usz, si))) return rc;
      if ((rc = ops->msm_pairs(c, si, groups[v], d_aff[v], d_aff[v] + ops->aff_words[groups[v]], counts[v] - 1, rlc_seed32, tweak,
                               d_pairs[v], err, errcap))) return rc;
    }
    c.mark("verify: msm launches enqueued");
    // 2b. CheckForCorrectness on the challenge, when asked for (the operator's default is No: the challenge is the output
    // of the previous verification): non-zero, and under Full on the curve and in the subgroup
    uint32_t* d_status_in = nullptr;
    if (check_input != CHECK_NO) {
      uint8_t* d_ch;
      if ((rc = c.alloc((void**)&d_ch, L.acc_size))) return rc;
      if ((rc = status_buffer(c, &d_status_in, 0, false, err, errcap))) return rc;
      CUDA_TRY(cudaMemcpyAsync(d_ch, challenge, L.acc_size, cudaMemcpyHostToDevice, c.s[0]));
      for (int v = 0; v < 5; v++) {
        if (counts[v] == 0) continue;
        if ((rc = ops->reencode(c, 0, groups[v], d_ch + L.off_u[v], 0, counts[v], nullptr, 0, check_input, check_input == CHECK_FULL ? 1u : 0u,
                                nullptr, d_status_in, err, errcap))) return rc;
      }
    }
    if ((rc = sync_all(c, err, errcap))) return rc;
    if (d_status_in && (rc = check_status(c, d_status_in, "challenge", err, errcap))) return rc == SSO_E_INPUT ? SSO_E_VERIFY : rc;
    if ((rc = check_status(c, d_status, "response", err, errcap))) return rc == SSO_E_INPUT ? SSO_E_VERIFY : rc;
    CUDA_TRY(cudaMemcpy(new_challenge + 64, d_new + 64, L.acc_size - 64, cudaMemcpyDeviceToHost));
    for (int v = 0; v < 4; v++) {
      if (!d_pairs[v]) continue;
      pairs[v].resize(2 * point_size(L.cs, groups[v], 0));
      CUDA_TRY(cudaMemcpy(pairs[v].data(), d_pairs[v], pairs[v].size(), cudaMemcpyDeviceToHost));
    }
    c.mark("verify: results D2H");
  } else {
    std::vector<RVec> vecs;
    if (check_input != CHECK_NO) {
      for (int v = 0; v < 5; v++)
        vecs.push_back({groups[v], challenge + L.off_u[v], 0, counts[v], nullptr, 0, 0, check_input, check_input == CHECK_FULL ? 1u : 0u, 0, inames[v]});
      if ((rc = stream_reencode(ops, L.cs, vecs, piece_elems, nullptr, 0, *P, nullptr, err, errcap))) return rc == SSO_E_INPUT ? SSO_E_VERIFY : rc;
      vecs.clear();
    }
    for (int v = 0; v < 5; v++)
      vecs.push_back({groups[v], response + L.off_c[v], 1, counts[v], new_challenge + L.off_u[v], 0, (ratio_check && v < 4) ? 1u : 0u,
                      elem_check, subgroup, TWEAK_P1_VERIFY | (uint64_t)v, vnames[v]});
    std::vector<std::vector<uint8_t>> out_pairs;
    if ((rc = stream_reencode(ops, L.cs, vecs, piece_elems, rlc_seed32, chunk_index, *P, &out_pairs, err, errcap))) return rc == SSO_E_INPUT ? SSO_E_VERIFY : rc;
    for (int v = 0; v < 4; v++) if (ratio_check && counts[v] >= 2) pairs[v] = out_pairs[v];
  }
  // 3. the side thread's results: hash chain (the response must continue the challenge; the new challenge's hash slot chains
  // the response), the validated public key and the g2_s points of the proofs
  side_thread.join();
  resp_hasher.join();
  if (ch_hash_out) memcpy(ch_hash_out, side.ch_hash, 64);
  if (memcmp(side.ch_hash, response, 64) != 0) { set_err(err, errcap, "hash chain broken: response does not continue the challenge"); return SSO_E_VERIFY; }
  if (side.rc != SSO_OK) { set_err(err, errcap, "%s", side.err); return side.rc; }
  memcpy(new_challenge, side.resp_hash, 64);
  const std::vector<uint8_t>& g2s = side.g2s;
  c.mark("verify: hashes, public key, hash_to_g2");
  // 5. collect the same_ratio checks
  std::vector<RatioCheck> checks;
  const uint8_t* pk_g2 = pk + 6 * g1u;                       // tau_g2, alpha_g2, beta_g2 (= g2_s_x)
  static const char* pok_names[3] = {"proof of knowledge: tau", "proof of knowledge: alpha", "proof of knowledge: beta"};
  for (int i = 0; i < 3; i++)
    add_check(checks, pok_names[i], pk + (size_t)2 * i * g1u, pk + (size_t)(2 * i + 1) * g1u, g1u, g2s.data() + (size_t)i * g2u,
              pk_g2 + (size_t)i * g2u, g2u);
  const uint8_t* after = new_challenge;
  if (chunk_index == 0 && L.on >= 2) {
    // element 0 must still be the generator; element 1 / alpha / beta must have moved by the proven scalars
    std::vector<uint8_t> gen(g1u + g2u);
    if ((rc = generator_bytes(c, ops, L.cs, curve, gen.data(), err, errcap))) return rc;
    if (memcmp(after + L.off_u[0], gen.data(), g1u) != 0) { set_err(err, errcap, "tau_g1[0] is not the G1 generator"); return SSO_E_VERIFY; }
    if (memcmp(after + L.off_u[1], gen.data() + g1u, g2u) != 0) { set_err(err, errcap, "tau_g2[0] is not the G2 generator"); return SSO_E_VERIFY; }
    add_check(checks, "before/after: tau_g1[1] vs tau proof", challenge + L.off_u[0] + g1u, after + L.off_u[0] + g1u, g1u,
              g2s.data(), pk_g2, g2u);
    add_check(checks, "before/after: alpha_g1[0] vs alpha proof", challenge + L.off_u[2], after + L.off_u[2], g1u,
              g2s.data() + g2u, pk_g2 + g2u, g2u);
    add_check(checks, "before/after: beta_g1[0] vs beta proof", challenge + L.off_u[3], after + L.off_u[3], g1u,
              g2s.data() + 2 * g2u, pk_g2 + 2 * g2u, g2u);
    add_check(checks, "before/after: beta_g2 vs beta_g1[0]", challenge + L.off_u[3], after + L.off_u[3], g1u,
              challenge + L.off_u[4], after + L.off_u[4], g2u);
  }
  if (ratio_check && !pairs[1].empty()) {
    // consecutive powers inside the chunk share one ratio: compare the G1 combinations with the G2 one.  A chunk past
    // 2^power holds tau_g1 only — no G2 element to compare with: its power ratios are checked on the combined accumulator
    // by transform_ratios ([UP]: Phase1::aggregate_verification; reference src/bin/verify_transcript.rs:811-822).
    const uint8_t* g2p = pairs[1].data();
    if (chunk_index == 0) g2p = after + L.off_u[1];           // (tau_g2[0], tau_g2[1]) exactly, as upstream
    if (!pairs[0].empty()) add_check(checks, "power ratio: tau_g1", pairs[0].data(), pairs[0].data() + g1u, g1u, g2p, g2p + g2u, g2u);
    if (!pairs[2].empty()) add_check(checks, "power ratio: alpha_g1", pairs[2].data(), pairs[2].data() + g1u, g1u, g2p, g2p + g2u, g2u);
    if (!pairs[3].empty()) add_check(checks, "power ratio: beta_g1", pairs[3].data(), pairs[3].data() + g1u, g1u, g2p, g2p + g2u, g2u);
    if (chunk_index == 0)
      add_check(checks, "power ratio: tau_g2", after + L.off_u[0], after + L.off_u[0] + g1u, g1u, pairs[1].data(), pairs[1].data() + g2u, g2u);
  }
  rc = run_checks(c, ops, checks, err, errcap);
  c.mark("verify: pairings");
  return rc;
}

// Work queue over the chunks of a batch: `host_threads` host workers, each running one chunk at a time through
// `one_chunk(index, device, err, errcap)`; device < 0 spreads the workers over all visible devices.
template <class Fn>
inline int32_t run_chunks_in_flight(size_t n_chunks, uint32_t host_threads, int device, char* err, size_t errcap, Fn one_chunk) {
  if (n_chunks == 0) return SSO_OK;
  int ndev = 1;
  if (device < 0) {
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { set_err(err, errcap, "no CUDA device available (this library has no CPU fallback)"); return SSO_E_CUDA; }
  }
  size_t workers = host_threads ? host_threads : (size_t)3 * ndev;
  if (workers > n_chunks) workers = n_chunks;
  if (workers > 64) workers = 64;
  std::atomic<size_t> next{0};
  std::atomic<int32_t> first_rc{SSO_OK};
  std::mutex err_lock;
  auto work = [&](size_t t) {
    char local[512];
    const int dev = device < 0 ? (int)(t % (size_t)ndev) : device;
    for (;;) {
      size_t i = next.fetch_add(1);
      if (i >= n_chunks || first_rc.load() != SSO_OK) return;
      local[0] = 0;
      int32_t rc = one_chunk(i, dev, local, sizeof(local));
      if (rc != SSO_OK) {
        std::lock_guard<std::mutex> g(err_lock);
        if (first_rc.load() == SSO_OK) {
          first_rc.store(rc);
          set_err(err, errcap, "chunk %zu of the batch: %s", i, local);
        }
        return;
      }
    }
  };
  std::vector<std::thread> pool;
  for (size_t t = 1; t < workers; t++) pool.emplace_back(work, t);
  work(0);
  for (auto& t : pool) t.join();
  return first_rc.load();
}


}  // namespace sso
